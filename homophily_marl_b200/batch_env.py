"""Batched, HBM-resident SSD env (Cleanup / Harvest): the tensor-level API.

``SSDBatchEnv`` owns B env instances on one B200.  State lives in PyTorch-owned
device tensors (packed u8 grids + one u32 per agent); every transition and every
observation is produced by the sm_100a kernels behind the C ABI
(``include/ssd_b200.h``).  PyTorch is only the allocator / stream provider here.

Replaces, batched: MapEnv.reset / step / get_obs / get_state
(src/envs/ssd/map_env.py:874-957, 986-993 of the reference).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _capi, mapspec


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise RuntimeError("homophily_marl_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"device must be a CUDA device, got {device!r}")
    return torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())


OBS_FORMATS = {"rgb": _capi.SSD_OBS_RGB, "index4": _capi.SSD_OBS_INDEX4}


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class SSDBatchEnv:
    def __init__(self, name, n_envs, num_agents, map="default", view_size=7, episode_limit=100,
                 extra_args=None, seed=0, device="cuda:0", env_gid_base=0, rows=None, params=None,
                 fire_cost=1, hit_penalty=0, want_state=False, check_actions=False, keep_episode_end=False, variants=None,
                 variant_of=None):
        # keep_episode_end: allocate end_obs_buf / end_state_buf / end_ep_ret_buf, which step / step_range with auto_reset fill
        #   with what an env whose episode ended saw before its reset
        # tag_timeout: steps an agent hit by a FIRE ray is out of play (off the map, action ignored, zero view); 0 = never
        # obs_format: "rgb" (u8 RGB planes, the reference's get_obs * 256) or "index4" (packed 4-bit colour indices)
        # state_format: the same choice for the state image (get_state * 256), independent of obs_format
        # variants (also extra_args["variants"]): per-env variants of this config, a list of mapspec.compile_variant override
        #   dicts ({} = this config); env b runs variant variant_of[b], by default (env_gid_base + b) % len(variants)
        # episode_stats: per-agent episode counters in stats_buf (and, with keep_episode_end, end_stats_buf), the inputs of
        #   social_metrics(); without it nothing is allocated and no kernel counts
        # reward_shaping: {"alpha", "beta", "decay", "prosocial"} (mapspec.reward_shaping), the inequity-averse / prosocial
        #   reward every step writes to shaped_buf (trace in shape_trace_buf); a variant dict may carry its own.  Without it (and
        #   without a variant's) nothing is allocated and no kernel runs
        extra = dict(random_spawn_point=False, random_spawn_rotation=0, disable_rotation_action=True,
                     disable_fire_action=True, obs_color="simplified", tag_timeout=0, obs_format="rgb", state_format="rgb",
                     episode_stats=False, reward_shaping=None)
        extra.update(extra_args or {})
        for key in ("obs_format", "state_format"):
            if extra[key] not in OBS_FORMATS:
                raise ValueError(f"{key} must be one of {sorted(OBS_FORMATS)}, got {extra[key]!r}")
        self.extra_args = extra
        shaping = None if extra["reward_shaping"] is None else mapspec.reward_shaping(extra["reward_shaping"])
        self.name = name
        self.spec = mapspec.compile_map(name, map, num_agents, view_size, episode_limit,
                                        obs_color=extra["obs_color"], rows=rows, params=params,
                                        fire_cost=fire_cost, hit_penalty=hit_penalty,
                                        tag_timeout=int(extra["tag_timeout"]))
        self.device = _require_cuda(device)
        # debug switch (one device sync per step): out-of-range action codes raise KeyError like the reference's action_map
        self.check_actions = bool(check_actions) or os.environ.get("SSD_B200_CHECK_ACTIONS") == "1"
        self.lib = _capi.load()
        s = self.spec
        self.B, self.n, self.H, self.W, self.G, self.N = int(n_envs), s.n_agents, s.H, s.W, s.G, s.N
        self.n_actions, self.episode_limit = s.n_actions, s.episode_limit
        self.seed, self.env_gid_base = int(seed), int(env_gid_base)

        cfg = _capi.SsdConfig()
        cfg.kind, cfg.n_envs, cfg.n_agents = s.kind, self.B, s.n_agents
        cfg.height, cfg.width, cfg.view, cfg.episode_limit = s.H, s.W, s.view, s.episode_limit
        cfg.fire_cost, cfg.hit_penalty, cfg.beam_len = s.fire_cost, s.hit_penalty, s.beam_len
        cfg.tag_timeout = s.tag_timeout
        cfg.random_spawn_point = int(bool(extra["random_spawn_point"]))
        rot = extra["random_spawn_rotation"]
        cfg.spawn_rotation = -1 if rot is None else int(rot)
        cfg.device = self.device.index
        cfg.seed, cfg.env_gid_base = self.seed & (2 ** 64 - 1), self.env_gid_base & 0xFFFFFFFF
        self._ascii = s.ascii_bytes()
        cfg.ascii_map = self._ascii
        self._thr_a = np.ascontiguousarray(s.thr_apple, dtype=np.uint32)
        self._thr_w = np.ascontiguousarray(s.thr_waste, dtype=np.uint32)
        cfg.n_waste_lut = len(self._thr_a)
        cfg.thr_apple, cfg.thr_waste = self._thr_a.ctypes.data, self._thr_w.ctypes.data
        for k in range(4):
            cfg.thr_harvest[k] = int(s.thr_harvest[k])
        for i in range(16):
            for ch in range(3):
                cfg.color_lut[i][ch] = int(s.lut[i, ch])
        self._h = C.c_void_p()
        _capi.check(self.lib.ssd_create(C.byref(cfg), C.byref(self._h)))
        lay = _capi.SsdLayout()
        _capi.check(self.lib.ssd_get_layout(self._h, C.byref(lay)))
        self.layout = lay
        assert lay.n_actions == self.n_actions and lay.n_cells == self.G
        self.obs_format, self.obs_layout = "rgb", self.get_obs_layout("rgb")
        if extra["obs_format"] != "rgb":
            self._set_format(extra["obs_format"])
        self.state_format, self.state_layout = "rgb", self.get_state_layout("rgb")
        if extra["state_format"] != "rgb":
            self._set_state_format(extra["state_format"])
        self.variant, self.variant_specs = None, [self.spec]
        variants = extra.get("variants") if variants is None else variants
        if variants is not None:
            self._set_variants(variants, variant_of)
        elif variant_of is not None:
            raise ValueError("variant_of needs variants")

        dev, B, n = self.device, self.B, self.n
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.grid_buf = z((B, lay.grid_stride), torch.uint8)
        self.agent_buf = z((B, lay.agent_stride), torch.int32)
        self.ep_ret_buf = z((B, lay.agent_stride), torch.int32)
        self.t_buf = z((B,), torch.int32)
        self.tick_buf = z((B,), torch.int32)
        self.counts_buf = z((B,), torch.int32)                 # #apple cells | #waste cells << 16 of every grid
        self.reward = z((B, n), torch.int8)
        self.clean = z((B, n), torch.uint8)
        self.apple_cnt = z((B,), torch.int16)
        self.done = z((B,), torch.uint8)
        self.keep_episode_end = bool(keep_episode_end)
        self.obs_buf = self.new_obs_buffer()
        self.end_obs_buf = self.new_obs_buffer() if self.keep_episode_end else None
        self.end_ep_ret_buf = z((B, lay.agent_stride), torch.int32) if self.keep_episode_end else None
        self.stats_buf = self.end_stats_buf = None
        if extra["episode_stats"]:
            self.stats_buf = z((B, _capi.SSD_N_STATS, lay.agent_stride), torch.int32)
            self.end_stats_buf = z((B, _capi.SSD_N_STATS, lay.agent_stride), torch.int32) if self.keep_episode_end else None
            _capi.check(self.lib.ssd_set_stats(self._h, _ptr(self.stats_buf), _ptr(self.end_stats_buf)))
        self.shape_trace_buf = self.shaped_buf = self.shaping_params = None
        if shaping is not None or any(sp.reward_shaping is not None for sp in self.variant_specs):
            # one parameter set per variant (ssd_set_reward_shaping): a variant's own, else the handle's, else the defaults
            shaping = shaping or mapspec.reward_shaping({})
            self.shaping_params = [shaping if sp.reward_shaping is None else sp.reward_shaping for sp in self.variant_specs]
            self.shape_trace_buf = z((B, lay.agent_stride), torch.float32)
            self.shaped_buf = z((B, lay.agent_stride), torch.float32)
            recs = (_capi.SsdShaping * len(self.shaping_params))(*[_capi.SsdShaping(*q) for q in self.shaping_params])
            _capi.check(self.lib.ssd_set_reward_shaping(self._h, len(recs), recs, _ptr(self.shape_trace_buf),
                                                        _ptr(self.shaped_buf)))
        self.want_state = bool(want_state)
        self._alloc_state()
        self._st = _capi.SsdState(*[t.data_ptr() for t in (self.grid_buf, self.agent_buf, self.ep_ret_buf,
                                                            self.t_buf, self.tick_buf, self.counts_buf)])
        self._keep = None

    # ------------------------------------------------------------------ per-env variants
    def _set_variants(self, variants, variant_of):
        """``ssd_set_variants`` with the compiled ``variants``, then ``ssd_set_env_variants`` with ``self.variant``."""
        specs = [mapspec.compile_variant(self.spec, v) for v in variants]
        if not 1 <= len(specs) <= _capi.SSD_MAX_VARIANTS:
            raise ValueError(f"variants needs 1..{_capi.SSD_MAX_VARIANTS} entries, got {len(specs)}")
        recs, keep = (_capi.SsdVariant * len(specs))(), []
        for r, sp in zip(recs, specs):
            a = sp.ascii_bytes()
            ta = np.ascontiguousarray(sp.thr_apple, dtype=np.uint32)
            tw = np.ascontiguousarray(sp.thr_waste, dtype=np.uint32)
            keep += [a, ta, tw]
            r.ascii_map, r.n_waste_lut, r.thr_apple, r.thr_waste = a, len(ta), ta.ctypes.data, tw.ctypes.data
            for k in range(4):
                r.thr_harvest[k] = int(sp.thr_harvest[k])
            r.fire_cost, r.hit_penalty, r.tag_timeout = sp.fire_cost, sp.hit_penalty, sp.tag_timeout
        if variant_of is None:
            variant_of = (np.arange(self.B, dtype=np.int64) + self.env_gid_base) % len(specs)
        ids = torch.as_tensor(np.asarray(variant_of.cpu() if torch.is_tensor(variant_of) else variant_of, dtype=np.int64))
        if ids.shape != (self.B,) or int(ids.min()) < 0 or int(ids.max()) >= len(specs):
            raise ValueError(f"variant_of must be [B] ids in 0..{len(specs) - 1}")
        _capi.check(self.lib.ssd_set_variants(self._h, len(specs), recs))
        # the kernels read this tensor in every later launch: write it (and reset the env for a new layout) to move an env
        self.variant = ids.to(device=self.device, dtype=torch.uint8).contiguous()
        _capi.check(self.lib.ssd_set_env_variants(self._h, _ptr(self.variant)))
        self.variant_specs = specs

    # ------------------------------------------------------------------ observation format
    def get_obs_layout(self, fmt):
        """``ssd_obs_layout`` (format, row_stride, plane_stride, agent_stride, env_stride) of "rgb" or "index4"."""
        lay = _capi.SsdObsLayout()
        _capi.check(self.lib.ssd_get_obs_layout(self._h, OBS_FORMATS[fmt], C.byref(lay)))
        return lay

    def _set_format(self, fmt):
        _capi.check(self.lib.ssd_set_obs_format(self._h, OBS_FORMATS[fmt]))
        self.obs_format, self.obs_layout = fmt, self.get_obs_layout(fmt)

    def set_obs_format(self, fmt):
        """Switches the format every later step / reset / render writes, and reallocates ``obs_buf`` for it.  Host-side: a
        CUDA graph captured before keeps the format it was captured with."""
        if fmt not in OBS_FORMATS:
            raise ValueError(f"obs_format must be one of {sorted(OBS_FORMATS)}, got {fmt!r}")
        self._set_format(fmt)
        self.extra_args["obs_format"] = fmt
        self.obs_buf = self.new_obs_buffer()
        if self.keep_episode_end:
            self.end_obs_buf = self.new_obs_buffer()

    # ------------------------------------------------------------------ state image format
    def get_state_layout(self, fmt):
        """``ssd_state_layout`` (format, row_stride, plane_stride, env_stride) of "rgb" or "index4"."""
        lay = _capi.SsdStateLayout()
        _capi.check(self.lib.ssd_get_state_layout(self._h, OBS_FORMATS[fmt], C.byref(lay)))
        return lay

    def _set_state_format(self, fmt):
        _capi.check(self.lib.ssd_set_state_format(self._h, OBS_FORMATS[fmt]))
        self.state_format, self.state_layout = fmt, self.get_state_layout(fmt)

    def _alloc_state(self):
        """``state_buf``: the state image buffer of the current format, u8 [B, 3, H, W] for RGB (also ``state_rgb``) or
        [B, env_stride] for index4 (``state_rgb`` is then None); both None without ``want_state``.  ``end_state_buf``, with
        ``keep_episode_end``, has the same shape."""
        self.state_buf = self.state_rgb = self.end_state_buf = None
        if self.want_state:
            shape = (self.B, 3, self.H, self.W) if self.state_format == "rgb" else (self.B, self.state_layout.env_stride)
            self.state_buf = torch.zeros(shape, dtype=torch.uint8, device=self.device)
            if self.state_format == "rgb":
                self.state_rgb = self.state_buf
            if self.keep_episode_end:
                self.end_state_buf = torch.zeros(shape, dtype=torch.uint8, device=self.device)

    def set_state_format(self, fmt):
        """Switches the format every later step / render writes the state image in, and reallocates ``state_buf``.
        Host-side: a CUDA graph captured before keeps the format it was captured with."""
        if fmt not in OBS_FORMATS:
            raise ValueError(f"state_format must be one of {sorted(OBS_FORMATS)}, got {fmt!r}")
        self._set_state_format(fmt)
        self.extra_args["state_format"] = fmt
        self._alloc_state()

    def _state_index4(self, what):
        if self.state_format != "index4" or self.state_buf is None:
            raise ValueError(f"{what} needs state_format 'index4' and want_state=True")

    def state_packed(self, buf=None):
        """[B, H, row_stride] u8 view (no copy) of an index4 state buffer: cell c of a row is byte c >> 1, low nibble when c
        is even."""
        self._state_index4("state_packed()")
        buf = self.state_buf if buf is None else buf
        lay = self.state_layout
        return buf.as_strided((self.B, self.H, lay.row_stride), (lay.env_stride, lay.row_stride, 1))

    def state_index(self, buf=None):
        """[B, H, W] u8 colour indices (unpacked copy): ``spec.lut[state_index()]`` is the RGB state image."""
        p = self.state_packed(buf)
        return torch.stack((p & 15, p >> 4), dim=-1).reshape(self.B, self.H, -1)[..., :self.W]

    def state_float(self, env_begin=0, env_count=None, buf=None, out=None):
        """f32 [env_count, 3, H, W] of envs [env_begin, env_begin + env_count) of an index4 state buffer (``state_buf`` by
        default, or ``end_state_buf``), through one ``ssd_expand_state`` launch on the current stream: bit-identical to
        ``state_rgb.float() / 256`` of an RGB env."""
        self._state_index4("state_float()")
        buf = self.state_buf if buf is None else buf
        env_count = self.B - env_begin if env_count is None else int(env_count)
        shape = (env_count, 3, self.H, self.W)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous() or tuple(out.shape) != shape:
            raise ValueError(f"out must be a contiguous float32 CUDA tensor of shape {shape}")
        if buf.dtype != torch.uint8 or not buf.is_cuda or buf.numel() < self.B * self.state_layout.env_stride:
            raise ValueError("buf must be a uint8 CUDA index4 state buffer of B * env_stride bytes")
        _capi.check(self.lib.ssd_expand_state(self._h, _ptr(buf), int(env_begin), env_count, _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ buffers / views
    def new_obs_buffer(self):
        """Flat u8 [B, env_stride] buffer in the layout of the current observation format."""
        return torch.zeros((self.B, self.obs_layout.env_stride), dtype=torch.uint8, device=self.device)

    def obs_view(self, buf=None):
        """[B, n, 3, N, N] u8 view (no copy) of an RGB obs buffer; ``view / 256`` equals get_obs()."""
        if self.obs_format != "rgb":
            raise ValueError("obs_view() reads RGB planes; this env writes index4 observations (use obs_index / obs_float)")
        buf = self.obs_buf if buf is None else buf
        lay = self.layout
        return buf.as_strided((self.B, self.n, 3, self.N, self.N),
                              (lay.obs_env_stride, lay.obs_agent_stride, lay.obs_plane_stride, lay.obs_row_stride, 1))

    def _index4(self, what):
        if self.obs_format != "index4":
            raise ValueError(f"{what} needs obs_format 'index4'")

    def obs_packed(self, buf=None):
        """[B, n, N, row_stride] u8 view (no copy) of an index4 buffer: pixel x of a row is byte x >> 1, low nibble when x is
        even."""
        self._index4("obs_packed()")
        buf = self.obs_buf if buf is None else buf
        lay = self.obs_layout
        return buf.as_strided((self.B, self.n, self.N, lay.row_stride), (lay.env_stride, lay.agent_stride, lay.row_stride, 1))

    def obs_index(self, buf=None):
        """[B, n, N, N] u8 colour indices (unpacked copy): ``spec.lut[obs_index()]`` is the RGB observation."""
        p = self.obs_packed(buf)
        return torch.stack((p & 15, p >> 4), dim=-1).reshape(self.B, self.n, self.N, -1)[..., :self.N]

    def obs_float(self, env_begin=0, env_count=None, buf=None, out=None):
        """f32 [env_count, n, 3, N, N] of envs [env_begin, env_begin + env_count) of an index4 buffer, through one
        ``ssd_expand_obs`` launch on the current stream: bit-identical to ``obs_view().float() / 256`` of an RGB env."""
        self._index4("obs_float()")
        buf = self.obs_buf if buf is None else buf
        env_count = self.B - env_begin if env_count is None else int(env_count)
        shape = (env_count, self.n, 3, self.N, self.N)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous() or tuple(out.shape) != shape:
            raise ValueError(f"out must be a contiguous float32 CUDA tensor of shape {shape}")
        if buf.dtype != torch.uint8 or not buf.is_cuda or buf.numel() < self.B * self.obs_layout.env_stride:
            raise ValueError("buf must be a uint8 CUDA index4 observation buffer of B * env_stride bytes")
        _capi.check(self.lib.ssd_expand_obs(self._h, _ptr(buf), int(env_begin), env_count, _ptr(out), self._stream()))
        return out

    @property
    def grid(self):
        return self.grid_buf[:, :self.G].view(self.B, self.H, self.W)

    @property
    def agent_pos(self):
        """[B, n, 2] (row, col) int32."""
        a = self.agent_buf[:, :self.n]
        return torch.stack([a & 0xFF, (a >> 8) & 0xFF], dim=-1)

    @property
    def agent_orient(self):
        return ((self.agent_buf[:, :self.n] >> 16) & 3).to(torch.uint8)

    @property
    def ep_ret(self):
        return self.ep_ret_buf[:, :self.n]

    @property
    def end_ep_ret(self):
        """[B, n] int32 episode returns written by an auto-reset step for the envs whose episode it ended (keep_episode_end)."""
        return None if self.end_ep_ret_buf is None else self.end_ep_ret_buf[:, :self.n]

    # ------------------------------------------------------------------ shaped rewards
    def shaped_reward(self):
        """[B, n] float32 view (no copy) of the shaped reward the last step wrote (extra_args ``reward_shaping``; DESIGN.md §3
        item 17): ``(w1*r_i + w*mean_j r_j - alpha/(n-1)*D_i) - beta/(n-1)*A_i``, with D_i / A_i the summed disadvantageous /
        advantageous gaps of the smoothed reward traces ``shape_trace_buf``."""
        if self.shaped_buf is None:
            raise ValueError("shaped_reward() needs extra_args reward_shaping (or a variant with its own)")
        return self.shaped_buf[:, :self.n]

    # ------------------------------------------------------------------ episode counters and social metrics
    def stats(self, buf=None):
        """[B, 7, n] int32 view (no copy) of the per-agent episode counters (``stats_buf``, or ``end_stats_buf``), field k being
        ``_capi.STAT_NAMES[k]``: apples eaten, sum of the 1-based step index t over them, FIREs, FIRE rays dealt that hit an agent,
        rays taken, steps started tagged out, waste cells cleaned; each counted since the env's last reset (extra_args
        ``episode_stats``)."""
        if self.stats_buf is None:
            raise ValueError("stats() needs extra_args episode_stats=True")
        return (self.stats_buf if buf is None else buf)[:, :, :self.n]

    def social_metrics(self, end=False):
        """Efficiency, equality, sustainability and peace (Perolat et al., 2017) of every env's current episode after ``t``
        steps, or with ``end=True`` of the episode an auto-reset step last finished (``end_stats_buf`` / ``end_ep_ret``, t =
        episode_limit; needs keep_episode_end).  A dict of fp64 [B] device tensors, computed without a host sync:
        efficiency = sum of ep_ret / t; equality = 1 - Gini of ep_ret, as the runners compute ``equality_metric`` (1 when the
        collective return is 0); sustainability = mean over the agents that ate of APPLE_T / APPLES (0 when none ate);
        peace = n - sum of OUT_STEPS / t.  An env at t = 0 has efficiency 0 and peace n."""
        if end:
            if self.end_stats_buf is None:
                raise ValueError("social_metrics(end=True) needs episode_stats and keep_episode_end")
            ret, st = self.end_ep_ret.double(), self.stats(self.end_stats_buf).double()
            t = torch.full((self.B,), float(self.episode_limit), dtype=torch.float64, device=self.device)
        else:
            ret, st = self.ep_ret.double(), self.stats().double()
            t = self.t_buf.double().clamp(min=1.0)
        coll = ret.sum(1)
        denom = 2 * self.n * ret.abs().sum(1)
        pair = (ret[:, None, :] - ret[:, :, None]).abs().sum((1, 2))
        equality = torch.where(coll != 0, 1 - pair / torch.where(denom == 0, 1.0, denom), 1.0)
        apples, apple_t = st[:, _capi.SSD_STAT_APPLES], st[:, _capi.SSD_STAT_APPLE_T]
        ate = apples > 0
        n_ate = ate.sum(1)
        per = torch.where(ate, apple_t / apples.clamp(min=1.0), 0.0)
        sustainability = torch.where(n_ate > 0, per.sum(1) / n_ate.clamp(min=1), 0.0)
        peace = self.n - st[:, _capi.SSD_STAT_OUT_STEPS].sum(1) / t
        return dict(efficiency=coll / t, equality=equality, sustainability=sustainability, peace=peace)

    @property
    def tag_out(self):
        """[B, n] u8: steps each agent is still tagged out (off the map); 0 = in play."""
        return ((self.agent_buf[:, :self.n] >> 24) & 0xFF).to(torch.uint8)

    def set_state(self, b, grid=None, pos_rc=None, orient=None):
        """Test/injection hook (SURVEY 5: get/set_state_tensors)."""
        if grid is not None:
            g = torch.as_tensor(np.asarray(grid, dtype=np.uint8).reshape(-1), device=self.device)
            self.grid_buf[b, :self.G] = g
            self._recount(slice(b, b + 1))
        if pos_rc is not None or orient is not None:
            a = self.agent_buf[b, :self.n].cpu().numpy().astype(np.int64)
            if pos_rc is not None:
                pr = np.asarray(pos_rc, dtype=np.int64)
                a = (a & ~0xFFFF) | pr[:, 0] | (pr[:, 1] << 8)
            if orient is not None:
                a = (a & ~0xFF0000) | (np.asarray(orient, dtype=np.int64) << 16)
            self.agent_buf[b, :self.n] = torch.as_tensor(a.astype(np.int32), device=self.device)

    def _recount(self, sel):
        """ssd_state.counts of the selected envs from their grids (needed after writing a grid directly)."""
        g = self.grid_buf[sel, :self.G]
        self.counts_buf[sel] = ((g == 2).sum(1) | ((g == 3).sum(1) << 16)).to(torch.int32)

    def load_state(self, grid=None, pos_rc=None, orient=None, t=None, tag_out=None):
        """Batched variant of ``set_state``: NumPy arrays [B,H,W] / [B,n,2] / [B,n] / [B]; ``tag_out`` [B,n] sets the
        tagging-out timers (non-zero only on envs whose variant has ``tag_timeout`` > 0)."""
        if grid is not None:
            g = np.ascontiguousarray(grid, dtype=np.uint8).reshape(self.B, self.G)
            self.grid_buf[:, :self.G] = torch.as_tensor(g, device=self.device)
            self._recount(slice(None))
        if tag_out is not None:
            tag_out = np.asarray(tag_out, dtype=np.int64)
            tags = np.array([sp.tag_timeout for sp in self.variant_specs])
            vid = np.zeros(self.B, dtype=np.int64) if self.variant is None else \
                np.minimum(self.variant.cpu().numpy().astype(np.int64), len(tags) - 1)
            if (tag_out.reshape(self.B, -1).any(1) & (tags[vid] == 0)).any():
                raise ValueError("tag_out needs tag_timeout > 0: with tag_timeout 0 the kernels ignore the timers")
            if tag_out.min(initial=0) < 0 or tag_out.max(initial=0) > 255:
                raise ValueError("tag_out must be in 0..255")
        if pos_rc is not None or orient is not None or tag_out is not None:
            a = self.agent_buf[:, :self.n].cpu().numpy().astype(np.int64)
            if pos_rc is not None:
                pr = np.asarray(pos_rc, dtype=np.int64)
                a = (a & ~0xFFFF) | pr[..., 0] | (pr[..., 1] << 8)
            if orient is not None:
                a = (a & ~0xFF0000) | (np.asarray(orient, dtype=np.int64) << 16)
            if tag_out is not None:
                a = (a & 0xFFFFFF) | (tag_out << 24)
            self.agent_buf[:, :self.n] = torch.as_tensor((a & 0xFFFFFFFF).astype(np.uint32).view(np.int32), device=self.device)
        if t is not None:
            self.t_buf.copy_(torch.as_tensor(np.asarray(t, dtype=np.int32), device=self.device))

    # ------------------------------------------------------------------ draws
    def _draws(self, draws):
        if not draws:
            return None
        keep = {}
        for k in ("prio", "u_apple", "u_waste", "wkey", "spawn_key"):
            v = draws.get(k)
            if v is not None:
                v = np.ascontiguousarray(v, dtype=np.uint32).view(np.int32)
                keep[k] = torch.as_tensor(v, device=self.device).contiguous()
        if draws.get("rot") is not None:
            keep["rot"] = torch.as_tensor(np.ascontiguousarray(draws["rot"], dtype=np.uint8), device=self.device)
        expect = dict(prio=self.B * self.n, u_apple=self.B * self.G, u_waste=self.B * self.G, wkey=self.B * self.G,
                      spawn_key=self.B * self.n * self.G, rot=self.B * self.n)
        for k, t in keep.items():
            if t.numel() != expect[k]:
                raise ValueError(f"draws[{k!r}] has {t.numel()} elements, expected {expect[k]}")
        self._keep = keep
        return _capi.SsdDraws(*[keep[k].data_ptr() if k in keep else None
                                for k in ("prio", "u_apple", "u_waste", "wkey", "spawn_key", "rot")])

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ entry points
    def reset(self, mask=None, draws=None, obs=True, obs_out=None):
        d = self._draws(draws)
        out = None if not obs else (self.obs_buf if obs_out is None else obs_out)
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        _capi.check(self.lib.ssd_reset(self._h, C.byref(self._st), _ptr(mask), C.byref(d) if d else None,
                                       _ptr(out), self._stream()))

    def _check_actions(self, actions):
        if actions.dtype != torch.uint8 or not actions.is_cuda or not actions.is_contiguous() or actions.numel() != self.B * self.n:
            raise ValueError("actions must be a contiguous uint8 CUDA tensor of shape [B, n]")
        if self.check_actions and bool((actions >= self.n_actions).any()):
            # the reference raises KeyError from action_map (agent.py:176,237); the kernel alone would treat the code as a no-op
            raise KeyError(int(actions.max()))

    def _step_out(self, obs_out, want_obs, want_state):
        return _capi.SsdStepOut(self.reward.data_ptr(), self.clean.data_ptr(), self.apple_cnt.data_ptr(),
                                self.done.data_ptr(),
                                (self.obs_buf if obs_out is None else obs_out).data_ptr() if want_obs else None,
                                self.state_buf.data_ptr() if (want_state and self.state_buf is not None) else None)

    def _episode_end(self, want_obs, want_state):
        if not self.keep_episode_end:
            return None
        return _capi.SsdEpisodeEnd(self.end_obs_buf.data_ptr() if want_obs else None,
                                   self.end_state_buf.data_ptr() if (want_state and self.end_state_buf is not None) else None,
                                   self.end_ep_ret_buf.data_ptr())

    def step(self, actions, draws=None, obs_out=None, want_obs=True, want_state=False, auto_reset=False):
        """actions: u8 CUDA tensor [B, n].  Results land in self.reward / clean / apple_cnt / done / obs.

        ``auto_reset=True`` (``ssd_step_autoreset``, one launch): every env whose ``done`` flag this step raised is reset in
        the same launch, and its slot of the observation buffer (and of the state image) then holds the FIRST observation of
        the new episode; ``done`` / ``reward`` keep the values of the finished step.  With ``keep_episode_end``, the finished
        step's observation, state image and ``ep_ret`` of those envs land in ``end_obs_buf`` / ``end_state_buf`` /
        ``end_ep_ret``; the slots of other envs are not written.  Envs may therefore run on different episode clocks
        (``load_state(t=...)``), which the reference -- one env, ``get_done()`` constantly False -- never needs."""
        if auto_reset:
            return self.step_range(actions, 0, self.B, draws, obs_out, want_obs, want_state, auto_reset=True)
        self._check_actions(actions)
        d = self._draws(draws)
        so = self._step_out(obs_out, want_obs, want_state)
        _capi.check(self.lib.ssd_step(self._h, C.byref(self._st), _ptr(actions), C.byref(d) if d else None,
                                      C.byref(so), self._stream()))

    def step_range(self, actions, env_begin, env_count, draws=None, obs_out=None, want_obs=True, want_state=False,
                   auto_reset=False):
        """``step`` restricted to envs [env_begin, env_begin + env_count) (``ssd_step_range``, or ``ssd_step_autoreset``
        with ``auto_reset``).  ``actions`` is the whole-batch [B, n] tensor; disjoint ranges may run concurrently on
        different CUDA streams (the launch goes to the caller's current stream), which lets one group's policy / logic
        overlap another group's observation stores."""
        self._check_actions(actions)
        d = self._draws(draws)
        so = self._step_out(obs_out, want_obs, want_state)
        if auto_reset:
            end = self._episode_end(want_obs, want_state)
            _capi.check(self.lib.ssd_step_autoreset(self._h, C.byref(self._st), _ptr(actions), C.byref(d) if d else None,
                                                    C.byref(so), C.byref(end) if end else None, int(env_begin),
                                                    int(env_count), self._stream()))
            return
        _capi.check(self.lib.ssd_step_range(self._h, C.byref(self._st), _ptr(actions), C.byref(d) if d else None,
                                            C.byref(so), int(env_begin), int(env_count), self._stream()))

    def render(self, obs_out=None, want_obs=True, want_state=False):
        o = (self.obs_buf if obs_out is None else obs_out) if want_obs else None
        s = self.state_buf if want_state else None
        _capi.check(self.lib.ssd_render(self._h, C.byref(self._st), _ptr(o), _ptr(s), self._stream()))

    def make_host_io(self, with_obs=True, with_state=False):
        """Pinned host mirrors for ``step_host`` (the reference-facing call with host buffers)."""
        pin = lambda t: torch.zeros(t.shape, dtype=t.dtype).pin_memory()  # noqa: E731
        io = dict(actions=torch.zeros((self.B, self.n), dtype=torch.uint8).pin_memory(),
                  reward=pin(self.reward), clean=pin(self.clean), apple_cnt=pin(self.apple_cnt), done=pin(self.done),
                  obs=pin(self.obs_buf) if with_obs else None,
                  state=pin(self.state_buf) if (with_state and self.state_buf is not None) else None,
                  agent=pin(self.agent_buf))
        io["d_actions"] = torch.zeros((self.B, self.n), dtype=torch.uint8, device=self.device)
        return io

    def step_host(self, io):
        """H2D actions -> step -> D2H reward/clean/apple_cnt/done(/obs/state) -> stream sync, all inside the C call."""
        want_state = io.get("state") is not None
        if want_state and self.state_buf is not None and io["state"].numel() != self.B * self.state_layout.env_stride:
            raise ValueError("io['state'] does not match the current state format: call make_host_io again after set_state_format")
        d_out = self._step_out(None, io["obs"] is not None, want_state)
        h_out = _capi.SsdStepOut(io["reward"].data_ptr(), io["clean"].data_ptr(), io["apple_cnt"].data_ptr(),
                                 io["done"].data_ptr(), io["obs"].data_ptr() if io["obs"] is not None else None,
                                 io["state"].data_ptr() if want_state else None)
        _capi.check(self.lib.ssd_step_host(self._h, C.byref(self._st), _ptr(io["actions"]), _ptr(io["d_actions"]),
                                           C.byref(d_out), C.byref(h_out), self._stream()))

    def pull_host(self, io, obs=True, state=True, agent=True):
        """Copies the current observation / state image / agent records into the pinned mirrors (one sync)."""
        if obs and io.get("obs") is not None:
            io["obs"].copy_(self.obs_buf, non_blocking=True)
        if state and io.get("state") is not None:
            self.render(want_obs=False, want_state=True)
            io["state"].copy_(self.state_buf, non_blocking=True)
        if agent:
            io["agent"].copy_(self.agent_buf, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()

    @property
    def launch_count(self):
        return int(self.lib.ssd_launch_count(self._h))

    def bytes_per_env_step(self):
        """ALGORITHMIC HBM bytes of one fused step+obs (SURVEY 8d): 2G + n(3N^2 + 11) + 3 for RGB, 2G + n(N ceil(N/2) + 11) + 3
        for index4."""
        obs = 3 * self.N * self.N if self.obs_format == "rgb" else self.N * ((self.N + 1) // 2)
        return 2 * self.G + self.n * (obs + 11) + 3

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.ssd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
