"""Shared scaffolding of the test suites: env and oracle factories over ``lockstep.CONFIGS``, random actions and draws, the
buffer and oracle comparisons, custom maps, the batched-runner stand-ins, the front-end helpers and ``env_var``.

A plain module, not a test file: test modules import shared code from here (or from ``lockstep`` and the ``*_ref`` /
``tag_oracle`` modules), never from each other."""
import contextlib
import os
import types

import numpy as np
import torch

import frontend_ref as R
import lockstep
from oracle import oracle as O
from tag_oracle import TagOracleBatch

DEV = "cuda:0"
FIRE, CLEAN = 7, 8
# the per-env state and step outputs two envs stepped with the same inputs must agree on
STATE = ("reward", "clean", "done", "apple_cnt", "grid_buf", "agent_buf", "ep_ret_buf", "t_buf", "tick_buf", "counts_buf")
BUFS = STATE + ("obs_buf", "state_buf")
END_BUFS = ("end_obs_buf", "end_state_buf", "end_ep_ret_buf")             # with keep_episode_end
COMBOS = [(o, s) for o in ("rgb", "index4") for s in ("rgb", "index4")]     # (obs_format, state_format)


@contextlib.contextmanager
def env_var(name, value):
    """Sets an environment variable for the body.  ``ssd_create`` reads SSD_B200_GENERIC and SSD_B200_PDL, so handles created
    inside take the setting for their whole life."""
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        yield
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


# ---------------------------------------------------------------------------------------------------- envs and oracles

def make_env(key, B, *, obs="rgb", state="rgb", color=None, T=0, seed=9, limit=1000, variants=None, spec=None,
             random_spawn=True, **kw):
    """An SSDBatchEnv of config ``key`` with want_state=True and, unless random_spawn=False, random spawn point and rotation.
    ``spec`` (a MapSpec of the same geometry, such as one of ``env.variant_specs``) supplies the layout, dynamics, FIRE costs
    and tag_timeout instead of the config and ``T``; ``kw`` goes to SSDBatchEnv."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    name, mp, n, view, c = lockstep.CONFIGS[key]
    extra = dict(obs_color=color or c, random_spawn_point=random_spawn, random_spawn_rotation=None if random_spawn else 0,
                 tag_timeout=T if spec is None else spec.tag_timeout, obs_format=obs, state_format=state)
    if spec is not None:
        kw.update(rows=spec.rows, params=spec.params, fire_cost=spec.fire_cost, hit_penalty=spec.hit_penalty)
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=limit, extra_args=extra, seed=seed, want_state=True,
                       variants=variants, **kw)


def make_ref(env, spec=None, seed=None):
    """The C oracle of ``env`` -- the tagging reference when the config tags -- with its size, seed, env ids and spawn rules.
    ``spec`` replaces the env's (a variant's MapSpec) and ``seed`` its seed."""
    spec = env.spec if spec is None else spec
    cls = TagOracleBatch if spec.tag_timeout else O.OracleBatch
    return cls.from_spec(spec, n_envs=env.B, seed=env.seed if seed is None else seed, env_gid0=env.env_gid_base,
                         random_spawn_point=bool(env.extra_args["random_spawn_point"]),
                         spawn_rotation=env.extra_args["random_spawn_rotation"])


def random_actions(rs, env, fire=0.0, clean=0.0):
    """[B, n] u8 actions, uniform over the env's action set; then FIRE with probability ``fire`` and, where the env has it,
    CLEAN with probability ``clean``.  A probability of 0 draws nothing from ``rs``."""
    a = rs.randint(0, env.n_actions, size=(env.B, env.n))
    if fire:
        a = np.where(rs.rand(env.B, env.n) < fire, FIRE, a)
    if clean and env.n_actions > CLEAN:
        a = np.where(rs.rand(env.B, env.n) < clean, CLEAN, a)
    return a.astype(np.uint8)


def random_draws(rs, env):
    """Every draw of one step (and of the resets it may do) for the whole batch, in the shapes ``step(draws=)`` takes."""
    B, n, G = env.B, env.n, env.G
    u = lambda *s: rs.randint(0, 2 ** 32, size=s, dtype=np.uint64).astype(np.uint32)  # noqa: E731
    return dict(prio=u(B, n), u_apple=u(B, G), u_waste=u(B, G), wkey=u(B, G), spawn_key=u(B, n * G),
                rot=rs.randint(0, 4, size=(B, n)).astype(np.uint8))


# ---------------------------------------------------------------------------------------------------- comparisons

def assert_same_buffers(a, b, keys, what):
    for k in keys:
        assert torch.equal(getattr(a, k), getattr(b, k)), (what, k)


def assert_state_matches_oracle(env, ora, what):
    """Grid, positions, orientations, episode returns, episode clocks and, with a tagging reference, the timers."""
    assert np.array_equal(env.grid.cpu().numpy(), ora.grid), (what, "grid")
    assert np.array_equal(env.agent_pos.cpu().numpy(), ora.pos_rc), (what, "pos")
    assert np.array_equal(env.agent_orient.cpu().numpy(), ora.orient), (what, "orient")
    assert np.array_equal(env.ep_ret.cpu().numpy(), ora.ep_ret), (what, "ep_ret")
    assert np.array_equal(env.t_buf.cpu().numpy(), ora.envs["t"]), (what, "t")
    if isinstance(ora, TagOracleBatch):
        assert np.array_equal(env.tag_out.cpu().numpy(), ora.tag_out), (what, "tag_out")


def assert_outputs_match_oracle(env, out, what):
    """The step outputs of ``env`` against the oracle's ``step`` result ``out`` (observations too, unless out["obs"] is None)."""
    for k in ("reward", "clean", "done"):
        assert np.array_equal(getattr(env, k).cpu().numpy(), out[k]), (what, k)
    assert np.array_equal(env.apple_cnt.cpu().numpy().view(np.uint16), out["apple_cnt"]), (what, "apple_cnt")
    if out.get("obs") is not None:
        got = env.obs_view().cpu().numpy()
        if not np.array_equal(got, out["obs"]):
            bad = np.argwhere(got != out["obs"])
            raise AssertionError((what, "obs", "first mismatch", bad[0].tolist(), len(bad), "bytes"))


def step_one_outputs(ora, actions, draws):
    """``ora.step_one`` on env 0 with injected draws, as the [1, ...] ``step`` result ``assert_outputs_match_oracle`` takes."""
    r, c, cnt, done = ora.step_one(actions, 0, {k: v.reshape(-1) for k, v in draws.items()})
    return dict(reward=r[None], clean=c[None], done=np.array([done], np.uint8), apple_cnt=np.array([cnt], np.uint16),
                obs=ora.obs_one(0)[None])


# ---------------------------------------------------------------------------------------------------- custom maps

def ssd_config(rows=("@@@@@", "@P B@", "@ P @", "@@@@@"), kind=0, n=1, view=7, **kw):
    """A C ``ssd_config`` for 4 envs on ``rows`` with flat threshold LUTs; ``kw`` sets further fields."""
    import ctypes as C
    from homophily_marl_b200 import _capi
    cfg = _capi.SsdConfig()
    cfg.kind, cfg.n_envs, cfg.n_agents, cfg.height, cfg.width, cfg.view = kind, 4, n, len(rows), len(rows[0]), view
    cfg.episode_limit, cfg.fire_cost, cfg.hit_penalty, cfg.beam_len = 10, 1, 0, 5
    cfg.ascii_map = "".join(rows).encode()
    thr = (C.c_uint32 * 8)()
    cfg.thr_apple = cfg.thr_waste = C.cast(thr, C.c_void_p)
    cfg.n_waste_lut = kw.pop("n_waste_lut", 1)
    for k, v in kw.items():
        setattr(cfg, k, v)
    cfg._keep = thr
    return cfg


def random_map(rs, kind, H, W, n_spawn):
    """Wall-enclosed random map in the reference alphabet with at least n_spawn 'P' cells."""
    g = np.full((H, W), " ", dtype="<U1")
    g[0, :] = g[-1, :] = "@"
    g[:, 0] = g[:, -1] = "@"
    inner = [(r, c) for r in range(1, H - 1) for c in range(1, W - 1)]
    rs.shuffle(inner)
    it = iter(inner)
    for _ in range(n_spawn):
        r, c = next(it)
        g[r, c] = "P"
    alphabet = ("B", "H", "R", "S", "@", " ", " ") if kind == "cleanup" else ("A", "A", "@", " ", " ", " ")
    for r, c in it:
        g[r, c] = alphabet[rs.randint(len(alphabet))]
    return ["".join(row) for row in g]


def custom_params(kind):
    from homophily_marl_b200 import mapspec
    if kind == "cleanup":
        return mapspec.EnvParams(mapspec.KIND_CLEANUP, "custom", 0.7, 0.1, 0.4, 0.25)
    return mapspec.EnvParams(mapspec.KIND_HARVEST, "custom", spawn_prob=(0.01, 0.1, 0.2, 0.4))


CUSTOM = [  # kind, H, W, n_agents, view, colour: odd views, both store paths, V = 31, 16 agents, 2 048 cells
    ("cleanup", 12, 11, 16, 3, "full"), ("cleanup", 20, 33, 7, 5, "simplified"), ("harvest", 16, 16, 16, 11, "full"),
    ("cleanup", 40, 50, 10, 9, "full"), ("harvest", 32, 64, 16, 31, "full"), ("harvest", 9, 38, 5, 13, "simplified"),
]


def make_custom_env(case, B, *, obs="rgb", state="rgb", T=0, seed=9):
    """An env on the random map of a CUSTOM-style case (seeded by its size), served by the runtime geometry."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    kind, H, W, n, view, color = case
    rows = random_map(np.random.RandomState(H * W + n), kind, H, W, n_spawn=min(32, n + 3))
    extra = dict(random_spawn_point=True, random_spawn_rotation=None, obs_color=color, tag_timeout=T, obs_format=obs,
                 state_format=state)
    return SSDBatchEnv(kind, B, n, view_size=view, episode_limit=1000, rows=rows, params=custom_params(kind), seed=seed,
                       extra_args=extra, want_state=True)


# ---------------------------------------------------------------------------------------------------- batched runner

class FakeBatch:
    """EpisodeBatch stand-in with the update() semantics of src/components/episode_buffer.py:87-116:
    per-key dtype, th.tensor() for non-tensors, clone for tensors, view_as into [B, T, ...] storage."""

    def __init__(self, scheme, B, T, device):
        self.scheme, self.batch_size, self.max_seq_length, self.device = scheme, B, T, device
        self.data = {k: torch.zeros((B, T) + tuple(v["shape"]), dtype=v.get("dtype", torch.float32), device=device)
                     for k, v in scheme.items()}
        self.data["filled"] = torch.zeros((B, T, 1), dtype=torch.long, device=device)

    def update(self, data, bs=slice(None), ts=slice(None)):
        ts = slice(ts, ts + 1) if isinstance(ts, int) else ts
        self.data["filled"][bs, ts] = 1
        for k, v in data.items():
            dtype = self.scheme[k].get("dtype", torch.float32)
            v = v.clone().detach() if isinstance(v, torch.Tensor) else torch.tensor(v, dtype=dtype, device=self.device)
            dest = self.data[k][bs, ts]
            self.data[k][bs, ts] = v.view_as(dest)

    def __getitem__(self, k):
        if isinstance(k, slice):                              # EpisodeBatch[lo:hi]: a view on the same storage
            view = FakeBatch.__new__(FakeBatch)
            view.scheme, view.max_seq_length, view.device = self.scheme, self.max_seq_length, self.device
            view.data = {name: t[k] for name, t in self.data.items()}
            view.batch_size, view.offset = view.data["filled"].shape[0], k.start or 0
            return view
        return self.data[k]


class ScriptedMAC:
    """Actions come from a fixed table (independent of the observations) so two runners can be compared."""

    def __init__(self, table, table_inc):
        self.table, self.table_inc = table, table_inc

    def init_hidden(self, batch_size):
        self.bs = batch_size

    def select_actions_env(self, batch, t_ep, t_env, test_mode=False):
        lo = getattr(batch, "offset", 0)
        return self.table[lo:lo + batch.batch_size, t_ep].clone()

    def select_actions_inc(self, actions, batch, t_ep, t_env, test_mode=False, agent_pos_replay=None):
        assert agent_pos_replay.shape[-1] == 2
        lo = getattr(batch, "offset", 0)
        return self.table_inc[lo:lo + batch.batch_size, t_ep].clone()


def _scheme(n, A, H, W, N):
    return {"state": {"shape": (3, H, W)}, "obs": {"shape": (n, 3, N, N)}, "actions": {"shape": (n, 1), "dtype": torch.long},
            "avail_actions": {"shape": (n, A), "dtype": torch.int}, "reward": {"shape": (n,)},
            "terminated": {"shape": (1,), "dtype": torch.uint8}, "clean_num": {"shape": (n,)}, "apple_den": {"shape": (n,)},
            "agent_pos": {"shape": (n, 2)}, "agent_orientation": {"shape": (n, 2)}, "actions_inc": {"shape": (n, n, 1), "dtype": torch.long}}


def make_runner(name="cleanup", mp="default3", n=3, view=7, B=6, T=9, groups=1, seed=3, extra=None, log_stat=None, **args):
    """A BatchedEpisodeRunner whose episodes land in FakeBatch: B envs, FIRE and rotation enabled, random spawn point and
    rotation, ``extra`` added to extra_args and ``args`` to the runner's args.  ``args.n_actions`` is set from the env."""
    from homophily_marl_b200.batched_runner import BatchedEpisodeRunner
    extra = dict(dict(random_spawn_point=True, random_spawn_rotation=None, disable_rotation_action=False,
                      disable_fire_action=False), **(extra or {}))
    env_args = dict(num_agents=n, render=False, episode_limit=T, is_replay=False, view_size=view, map=mp, extra_args=extra,
                    seed=seed)
    ns = types.SimpleNamespace(batch_size_run=B, env=name, env_args=env_args, device=DEV, name="homophily", mac="homophily_mac",
                               n_actions=None, ind_reward=True, runner_log_interval=10 ** 9, test_nepisode=B, env_groups=groups,
                               **args)
    runner = BatchedEpisodeRunner(ns, types.SimpleNamespace(log_stat=log_stat or (lambda k, v, t: None)))
    e = runner.env
    ns.n_actions = e.n_actions
    scheme = _scheme(n, e.n_actions, e.H, e.W, e.N)
    runner.use_batch_factory(lambda: FakeBatch(scheme, B, T + 1, e.device))
    return runner


def action_tables(runner, seed, high=None):
    """Random [B, T+1, n, 1] action and [B, T+1, n, n, 1] incentive tables for a scripted episode (actions below ``high``,
    by default n_actions), on the runner's device."""
    e = runner.env
    g = torch.Generator().manual_seed(seed)
    shape = (e.B, runner.episode_limit + 1, e.n)
    table = torch.randint(0, high or e.n_actions, shape + (1,), generator=g).to(e.device)
    table_inc = torch.randint(0, 3, shape + (e.n, 1), generator=g).to(e.device)
    return table, table_inc


def feature_mac(module, N, n, table, table_inc):
    """A MAC with scripted actions whose observations go through ``agent.rgb_preprocess`` = ``module`` (the fused front end
    serves that call when the runner has one)."""
    class Agent:
        conv_to_fc = module

        def rgb_preprocess(self, x):
            return module(x)

    class MAC:
        agent = Agent()

        def init_hidden(self, batch_size):
            pass

        def select_actions_env(self, batch, t_ep, t_env, test_mode=False):
            feats = self.agent.rgb_preprocess(batch["obs"][:, t_ep].reshape(-1, 3, N, N))
            assert feats.shape == (batch.batch_size * n, 32)
            return table[batch.offset:batch.offset + batch.batch_size, t_ep].clone()

        def select_actions_inc(self, actions, batch, t_ep, t_env, test_mode=False, agent_pos_replay=None):
            return table_inc[batch.offset:batch.offset + batch.batch_size, t_ep].clone()
    return MAC()


def _cfg(**kw):
    """The reference's run config for Cleanup default3 (baseline/refloop.py), with ``kw`` on top."""
    from baseline import refloop
    base = dict(seed=3, use_cuda=True, save_model=False, t_max=300, batch_size=4, buffer_size=16, test_nepisode=2,
                test_interval=10 ** 9, log_interval=10 ** 9, runner_log_interval=10 ** 9, learner_log_interval=1,
                env_args=dict(num_agents=3, map="default3"))
    base.update(kw)
    seed = base.pop("seed")
    return refloop.load_config("cleanup", seed=seed, **base)


# ---------------------------------------------------------------------------------------------------- fused front end

def _weights(view, seed, conv_scale=1.0, fc_scale=1.0):
    """conv_w, conv_b, fc_w, fc_b as float32 numpy arrays (PyTorch's default init of the reference module)."""
    torch.manual_seed(seed)
    P = 2 * view - 1
    conv, fc = torch.nn.Conv2d(3, 6, 3, 1), torch.nn.Linear(6 * P * P, 32)
    w = [t.detach().numpy().astype(np.float32).copy() for t in (conv.weight, conv.bias, fc.weight, fc.bias)]
    w[0] *= np.float32(conv_scale)
    w[2] *= np.float32(fc_scale)
    return w


def _front_end(w, view, slope=0.01):
    from homophily_marl_b200.frontend import ObsFrontEnd
    return ObsFrontEnd(*w, view, negative_slope=slope, device=DEV)


def _expect(case, view, got, host, rows, lay, w, slope, hi_check=True, scale="y"):
    """Asserts the bound on `got` (numpy [rows, 32]) and, with hi_check, that the hi-only FC misses it by >= 10x.

    scale="M" measures the error against 1 + M, M = |fc_b| + sum |W||a| the condition scale of the FC sum, instead of
    1 + |y|: with trained-like weights the sum cancels (M / (1 + |y|) reaches ~1 000 at 16x the default init) and no fp32
    contraction meets the 1 + |y| form there -- torch's own fp32 matmul of the exact activations measures 2.2e-5."""
    slope = float(np.float32(slope))                          # the kernel's slope is the float32 one
    y, M = R.forward64(host, rows, lay["AS"], lay["PS"], lay["RP"], view, *w, slope)
    tol = R.tolerance(view)

    def rel(v):
        return float((np.abs(np.asarray(v, np.float64) - y) / (1 + (M if scale == "M" else np.abs(y)))).max()) if y.size else 0.0
    err = rel(got)
    herr = rel(R.forward64_hi_only(host, rows, lay["AS"], lay["PS"], lay["RP"], view, *w, slope)) if hi_check else float("nan")
    print(f"frontend-err {case} V={view} err={err:.3e} tol={tol:.2e} hi_only={herr:.3e}"
          + (f" scale=1+M (vs 1+|y|: {R.rel_err(got, y):.3e})" if scale == "M" else ""))
    assert np.isfinite(got).all(), case
    assert err <= tol, (case, view, err, tol)
    if hi_check:
        assert herr >= 10 * tol, (case, view, herr, tol)
    return y


def _auto_grid(view, rows):
    """The grid ssd_frontend_forward picks without SSD_B200_FRONTEND_GRID (restated), and the number of (tile, chunk) units."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    P = 2 * view - 1
    n_chunks, tiles = P * ((P + 15) // 16), -(-rows // 128)
    units = tiles * n_chunks
    grid = min(units, sms)
    share = units / grid
    best = share + 1.5 * (2.0 if share < n_chunks else float(int(share / n_chunks) + 2))
    for s in range(1, n_chunks + 1):
        if tiles * s > sms:
            break
        cost = (n_chunks + s - 1) // s + 1.5
        if cost < best - 1e-9:
            best, grid = cost, tiles * s
    return grid, units
