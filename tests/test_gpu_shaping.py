"""GPU suite: shaped rewards (extra_args reward_shaping, ``ssd_set_reward_shaping``; DESIGN.md §3 item 17).

After every step the shaped rewards and traces equal, bit for bit, the NumPy float32 restatement (tests/shaping_ref.py) applied
to the GPU's own rewards, done flags and variant ids -- on every shipped config with and without tagging, under Philox and
injected draws, at 65 536 envs, on the runtime geometry and a custom map.  A handle with shaping is bit-identical to its twin
without it in every other buffer; a sweep of 8 parameter sets in one batch equals 8 single-parameter handles; env ranges on 8
streams (with and without programmatic dependent launch), auto-reset, masked reset, ssd_step_host and CUDA graphs keep the traces
right; and the batched runner and the PyMARL facade hand the shaped rewards to the learner while their statistics stay extrinsic."""
import ctypes as C
import math

import numpy as np
import pytest

import lockstep
from harness import (BUFS, COMBOS, CUSTOM, END_BUFS, FakeBatch, ScriptedMAC, _scheme, action_tables, assert_same_buffers,
                     custom_params, env_var, make_runner, random_actions, random_draws, random_map)
from shaping_ref import ShapingRef

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
HUGHES = {"alpha": 5.0, "beta": 0.05, "prosocial": 0.25}       # Hughes' Cleanup weights, mixed with some prosocial reward
SWEEP = [{"alpha": a, "beta": b, "decay": d, "prosocial": w}
         for a, b, d, w in ((0, 0, 0.5, 0), (5, 0.05, 0.96525, 0), (0, 5, 0.9, 0), (1, 1, 1.0, 0.5), (0.3, 0.7, 0.0, 1.0),
                            (12, 0, 0.99, 0.1), (0, 0, 0.96525, 0.75), (2.5, 2.5, 0.75, 0.25))]


def make(key, B, *, shaping=HUGHES, obs="rgb", state="rgb", T=0, seed=9, limit=1000, stats=False, **kw):
    """An SSDBatchEnv of config ``key`` (random spawn point and rotation, want_state) with shaping ``shaping`` (None: off)."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    name, mp, n, view, c = lockstep.CONFIGS[key]
    extra = dict(obs_color=c, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=T, obs_format=obs,
                 state_format=state, episode_stats=stats, reward_shaping=shaping)
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=limit, extra_args=extra, seed=seed, want_state=True, **kw)


def make_ref(env):
    var = None if env.variant is None else env.variant.cpu().numpy()
    return ShapingRef(env.B, env.n, env.shaping_params, var)


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def assert_matches(env, ref, what):
    """shaped and trace of ``env`` equal the restatement bit for bit (the pad lanes stay 0)."""
    for name, got, want in (("shaped", env.shaped_buf, ref.shaped), ("trace", env.shape_trace_buf, ref.trace)):
        g = got.cpu().numpy()
        assert not g[:, env.n:].any(), (what, name, "pad")
        g = g[:, :env.n]
        if not np.array_equal(bits(g), bits(want)):
            bad = np.argwhere(bits(g) != bits(want))[0]
            raise AssertionError((what, name, bad.tolist(), float(g[tuple(bad)]), float(want[tuple(bad)])))


def step_both(env, ref, at, auto_reset=False, **kw):
    env.step(at, auto_reset=auto_reset, **kw)
    ref.step(env.reward.cpu().numpy(), done=env.done.cpu().numpy() if auto_reset else None)


@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
@pytest.mark.parametrize("T", [0, 3])
def test_shaped_rewards_match_the_restatement(key, T):
    env = make(key, 16, T=T, limit=30)
    ref = make_ref(env)
    env.reset()
    rs = np.random.RandomState(10 * sorted(lockstep.CONFIGS).index(key) + T)
    for t in range(40):
        at = torch.as_tensor(random_actions(rs, env, fire=0.3, clean=0.3), device=env.device)
        if t < 25:
            step_both(env, ref, at, auto_reset=t % 5 == 4)
        else:                                                 # injected draws
            step_both(env, ref, at, draws=random_draws(rs, env), want_obs=False)
        assert_matches(env, ref, (key, T, t))
    assert (env.reward != 0).any() and (ref.trace != 0).any() and not np.array_equal(ref.shaped, env.reward.cpu().numpy())


@pytest.mark.parametrize("obs,state", COMBOS)
@pytest.mark.parametrize("stats,variants", [(False, False), (True, True)])
def test_shaping_changes_no_other_byte(obs, state, stats, variants):
    """A handle with shaping and its twin without agree in every buffer and pad byte over steps, ranges, auto-reset steps with
    episode-end buffers, masked resets, renders and host steps."""
    key, T = ("cleanup5", 3) if variants else ("harvest5", 3)
    var = [{}, {"fire_cost": 0, "hit_penalty": 1}, {"tag_timeout": 4, "reward_shaping": {"beta": 2.0}}] if variants else None
    a_env = make(key, 64, T=T, obs=obs, state=state, limit=12, keep_episode_end=True, stats=stats, variants=var)
    b_env = make(key, 64, T=T, obs=obs, state=state, limit=12, keep_episode_end=True, stats=stats, shaping=None,
                 variants=[{k: v for k, v in d.items() if k != "reward_shaping"} for d in var] if variants else None)
    assert b_env.shaped_buf is None and b_env.shape_trace_buf is None and b_env.shaping_params is None
    ref = make_ref(a_env)
    rs = np.random.RandomState(4)
    t0 = rs.randint(0, 12, size=64)
    for e in (a_env, b_env):
        e.reset()
        e.load_state(t=t0)
    keys = BUFS + END_BUFS + (("stats_buf", "end_stats_buf") if stats else ())
    for t in range(30):
        a = random_actions(rs, a_env, fire=0.3, clean=0.2)
        at = torch.as_tensor(a, device=a_env.device)
        mode = t % 5
        for e in (a_env, b_env):
            if mode == 0:
                e.step(at, want_state=True)
            elif mode == 1:
                e.step(at, want_state=True, auto_reset=True)
            elif mode == 2:
                e.step_range(at, 0, 40, want_state=True, auto_reset=True)
                e.step_range(at, 40, 24, want_state=True)
            elif mode == 3:
                e.reset(mask=torch.as_tensor(t0 % 3 == t % 3, device=e.device))
                e.render(want_obs=True, want_state=True)
            else:
                io = e.make_host_io()
                io["actions"].copy_(torch.as_tensor(a))
                e.step_host(io)
        r, d = a_env.reward.cpu().numpy(), a_env.done.cpu().numpy()
        if mode in (0, 4):
            ref.step(r)
        elif mode == 1:
            ref.step(r, done=d)
        elif mode == 2:
            ref.step(r, done=d, envs=slice(0, 40))
            ref.step(r, envs=slice(40, 64))
        else:
            ref.reset(t0 % 3 == t % 3)
        assert_same_buffers(a_env, b_env, keys, (obs, state, stats, variants, t))
        assert_matches(a_env, ref, (obs, state, stats, variants, t))
    a_env.close()
    b_env.close()


def test_sweep_of_8_parameter_sets_equals_single_parameter_handles():
    """One batch whose 8 variants differ only in their reward_shaping equals, env for env, 8 handles of one parameter set each."""
    mixed = make("cleanup5", 256, variants=[{"reward_shaping": s} for s in SWEEP], limit=20)
    twins = [make("cleanup5", 256, shaping=s, limit=20) for s in SWEEP]
    assert len(mixed.shaping_params) == 8 and mixed.shaping_params[1] == twins[1].shaping_params[0]
    vid = mixed.variant.cpu().numpy()
    ref = make_ref(mixed)
    rs = np.random.RandomState(7)
    for e in [mixed] + twins:
        e.reset()
    for t in range(30):
        at = torch.as_tensor(random_actions(rs, mixed, fire=0.3, clean=0.3), device=mixed.device)
        for e in [mixed] + twins:
            e.step(at, auto_reset=True)
        ref.step(mixed.reward.cpu().numpy(), done=mixed.done.cpu().numpy())
        assert_matches(mixed, ref, t)
        got_u, got_e = bits(mixed.shaped_reward().cpu().numpy()), bits(mixed.shape_trace_buf.cpu().numpy())
        for v, tw in enumerate(twins):
            m = vid == v
            assert np.array_equal(got_u[m], bits(tw.shaped_reward().cpu().numpy())[m]), (t, v)
            assert np.array_equal(got_e[m], bits(tw.shape_trace_buf.cpu().numpy())[m]), (t, v)
    u = mixed.shaped_reward().cpu().numpy()
    assert len({u[vid == v].tobytes() for v in range(8)}) == 8


@pytest.mark.parametrize("pdl", ["1", "0"])
def test_ranges_on_eight_streams(pdl):
    """8 env ranges of 512 envs on 8 streams (with and without programmatic dependent launch) shape what one whole-batch launch
    shapes, with auto-reset steps among them."""
    with env_var("SSD_B200_PDL", pdl):
        whole, parts = make("harvest5", 4096, T=3, limit=10), make("harvest5", 4096, T=3, limit=10)
    streams = [torch.cuda.Stream(device=parts.device) for _ in range(8)]
    rs = np.random.RandomState(3)
    ref = make_ref(whole)
    for e in (whole, parts):
        e.reset()
        e.load_state(t=np.random.RandomState(1).randint(0, 10, size=4096))
    torch.cuda.synchronize()
    for t in range(24):
        at = torch.as_tensor(random_actions(rs, whole, fire=0.4), device=whole.device)
        ar = t % 3 == 2
        step_both(whole, ref, at, auto_reset=ar)
        main = torch.cuda.current_stream(parts.device)
        for k, s in enumerate(streams):
            s.wait_stream(main)
            with torch.cuda.stream(s):
                parts.step_range(at, 512 * k, 512, auto_reset=ar)
        for s in streams:
            main.wait_stream(s)
        assert_same_buffers(whole, parts, BUFS + ("shaped_buf", "shape_trace_buf"), (pdl, t))
        assert_matches(parts, ref, (pdl, t))


@pytest.mark.parametrize("key,T", [("cleanup5", 0), ("harvest5", 3)])
def test_autoreset_writes_the_finished_step_then_zeroes_the_trace(key, T):
    """ssd_step_autoreset: the shaped reward of the finished step equals that of a step-then-masked-reset sequence, and the trace
    of every env it reset is 0 afterwards, as the sequence's reset leaves it."""
    fused, seq = make(key, 128, T=T, limit=10), make(key, 128, T=T, limit=10)
    rs = np.random.RandomState(6)
    t0 = rs.randint(0, 10, size=128)
    for e in (fused, seq):
        e.reset()
        e.load_state(t=t0)
    ended = 0
    for t in range(25):
        at = torch.as_tensor(random_actions(rs, fused, fire=0.4, clean=0.3), device=fused.device)
        fused.step(at, auto_reset=True)
        seq.step(at)
        d = seq.done.bool()
        assert torch.equal(fused.shaped_buf, seq.shaped_buf), t
        seq.reset(mask=d)
        assert torch.equal(fused.shape_trace_buf, seq.shape_trace_buf), t
        assert not fused.shape_trace_buf[d].any()
        ended += int(d.sum())
    assert ended > 0 and fused.shape_trace_buf.any()


def test_masked_reset_render_and_host_step():
    env = make("cleanup5", 256, T=3)
    env.reset()
    rs = np.random.RandomState(5)
    for _ in range(10):
        env.step(torch.as_tensor(random_actions(rs, env, fire=0.4, clean=0.3), device=env.device))
    before = env.shape_trace_buf.clone()
    mask = torch.as_tensor(rs.rand(256) < 0.4, device=env.device)
    launches = env.launch_count
    env.reset(mask=mask)
    torch.cuda.synchronize()
    assert env.launch_count == launches + 2                     # the reset kernel and the trace reset
    assert not env.shape_trace_buf[mask].any()
    assert torch.equal(env.shape_trace_buf[~mask], before[~mask]) and before[~mask].any()
    plain = make("cleanup5", 4, shaping=None)
    launches = plain.launch_count
    plain.reset()
    plain.step(torch.zeros((4, plain.n), dtype=torch.uint8, device=plain.device))
    assert plain.launch_count == launches + 2                   # no shaping: one reset and one step launch, nothing else
    # ssd_render leaves both buffers alone; ssd_step_host updates them as ssd_step does
    u, e = env.shaped_buf.clone(), env.shape_trace_buf.clone()
    env.render(want_obs=True, want_state=True)
    assert torch.equal(env.shaped_buf, u) and torch.equal(env.shape_trace_buf, e)
    twin = make("cleanup5", 256, T=3)
    twin.reset()
    for name in ("grid_buf", "agent_buf", "ep_ret_buf", "t_buf", "tick_buf", "counts_buf", "shape_trace_buf"):
        getattr(twin, name).copy_(getattr(env, name))
    a = torch.as_tensor(random_actions(rs, env, fire=0.4), device=env.device)
    io = env.make_host_io()
    io["actions"].copy_(a.cpu())
    launches = env.launch_count
    env.step_host(io)
    assert env.launch_count == launches + 2
    twin.step(a)
    torch.cuda.synchronize()
    assert_same_buffers(env, twin, ("reward", "shaped_buf", "shape_trace_buf"), "step_host")
    assert not torch.equal(env.shaped_buf, u)


def test_cuda_graph_capture_and_replay():
    eager, graphed = make("harvest5", 512, T=3, limit=7), make("harvest5", 512, T=3, limit=7)   # 16 steps: 2 resets, then 2 more
    rs = np.random.RandomState(9)
    acts = [torch.as_tensor(random_actions(rs, eager, fire=0.4), device=eager.device) for _ in range(5)]
    for e in (eager, graphed):
        e.reset()
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=graphed.device)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.step(acts[0], auto_reset=True)                # warm-up outside the capture, stepped like any step
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for a in acts:
                graphed.step(a, auto_reset=True)
    eager.step(acts[0], auto_reset=True)
    for _ in range(3):
        g.replay()
        for a in acts:
            eager.step(a, auto_reset=True)
    torch.cuda.synchronize()
    assert_same_buffers(eager, graphed, BUFS + ("shaped_buf", "shape_trace_buf"), "graph")
    assert graphed.shape_trace_buf.any() and graphed.shaped_buf.any()


def test_65536_envs():
    env = make("cleanup5", 65536, limit=8, shaping={"alpha": 5.0, "beta": 0.05})
    ref = make_ref(env)
    env.reset()
    rs = np.random.RandomState(2)
    for t in range(12):
        at = torch.as_tensor(random_actions(rs, env, fire=0.3, clean=0.3), device=env.device)
        step_both(env, ref, at, auto_reset=True, want_obs=False)
        assert_matches(env, ref, t)


def test_runtime_geometry_and_custom_map():
    with env_var("SSD_B200_GENERIC", "1"):
        env = make("harvest5", 32, T=3, limit=12)
    ref = make_ref(env)
    env.reset()
    rs = np.random.RandomState(8)
    for t in range(20):
        step_both(env, ref, torch.as_tensor(random_actions(rs, env, fire=0.3), device=env.device), auto_reset=t % 2 == 1)
        assert_matches(env, ref, ("generic", t))
    from homophily_marl_b200.batch_env import SSDBatchEnv
    for case in (CUSTOM[0], CUSTOM[4]):
        kind, H, W, n, view, color = case
        rows = random_map(np.random.RandomState(H * W + n), kind, H, W, n_spawn=min(32, n + 3))
        extra = dict(random_spawn_point=True, random_spawn_rotation=None, obs_color=color, tag_timeout=3, reward_shaping=HUGHES)
        env = SSDBatchEnv(kind, 16, n, view_size=view, episode_limit=1000, rows=rows, params=custom_params(kind), seed=9,
                          extra_args=extra, want_state=True)
        ref = make_ref(env)
        env.reset()
        for t in range(15):
            step_both(env, ref, torch.as_tensor(random_actions(rs, env, fire=0.4, clean=0.3), device=env.device))
            assert_matches(env, ref, (case, t))
        assert (ref.trace != 0).any()
        env.close()


def test_validation_on_a_handle():
    """Every refusal of ssd_set_reward_shaping on a real handle returns SSD_ERR_INVALID before any CUDA call and changes nothing;
    n_params = 0 with NULL, NULL turns shaping off."""
    from homophily_marl_b200 import _capi
    env = make("cleanup5", 8)
    lib, h = env.lib, env._h
    p = C.c_void_p(env.shaped_buf.data_ptr())
    ok = (_capi.SsdShaping * 1)(_capi.SsdShaping(1.0, 1.0, 0.5, 0.5))
    bad = [(1, (_capi.SsdShaping * 1)(_capi.SsdShaping(*q)), p, p) for q in
           ((math.nan, 0, 0.5, 0), (0, math.inf, 0.5, 0), (-1, 0, 0.5, 0), (0, -0.1, 0.5, 0), (0, 0, 1.01, 0), (0, 0, -0.5, 0),
            (0, 0, 0.5, 1.5), (0, 0, 0.5, -0.1), (0, 0, math.nan, 0))]
    bad += [(1, ok, p, None), (1, ok, None, p), (1, None, p, p), (0, None, p, p), (1, ok, None, None), (257, ok, p, p), (-1, ok, p, p)]
    env.reset()
    env.step(torch.ones((8, env.n), dtype=torch.uint8, device=env.device))
    torch.cuda.synchronize()
    before = lib.ssd_last_cuda_error()
    for n, params, tr, sh in bad:
        assert lib.ssd_set_reward_shaping(h, n, params, tr, sh) == _capi.SSD_ERR_INVALID, n
    assert lib.ssd_last_cuda_error() == before
    launches = env.launch_count
    env.step(torch.ones((8, env.n), dtype=torch.uint8, device=env.device))   # the handle still shapes, with its own parameters
    assert env.launch_count == launches + 2
    last = env.shaped_buf.clone()
    assert lib.ssd_set_reward_shaping(h, 0, None, None, None) == _capi.SSD_OK
    launches = env.launch_count
    env.step(torch.ones((8, env.n), dtype=torch.uint8, device=env.device))
    assert env.launch_count == launches + 1 and torch.equal(env.shaped_buf, last)
    env.close()


def test_batched_runner_shaped_return_equals_facade_episodes():
    """The runner's batch["reward"] is the shaped reward (summed without ind_reward); its statistics stay extrinsic and equal those
    of a runner without shaping; shaped_return and v{k}_shaped_return equal the facade's episodes env for env."""
    from homophily_marl_b200 import REGISTRY
    B, T, n = 6, 9, 3
    variants = [{}, {"reward_shaping": {"beta": 3.0, "prosocial": 0.5}}]
    runs = {}
    for shaped in (False, True):
        logged = {}
        extra = dict(obs_color="full", variants=variants if shaped else [{}, {}])
        if shaped:
            extra["reward_shaping"] = HUGHES
        runner = make_runner("cleanup", "default3", n, 7, B=B, T=T, groups=1, extra=extra,
                             log_stat=lambda k, v, t, logged=logged: logged.__setitem__(k, v))
        table, table_inc = action_tables(runner, 1)
        runner.mac = ScriptedMAC(table, table_inc)
        batch = runner.run(test_mode=True)
        runs[shaped] = (runner, logged, batch)
    (plain, plog, pbatch), (runner, logged, batch) = runs[False], runs[True]
    for k in ("test_return_mean", "test_collective_return_mean", "test_equality_metric_mean", "test_v1_return_mean"):
        assert logged[k] == plog[k], k
    assert "test_shaped_return_mean" not in plog and "shaped_return" not in plain.last_env_info
    extrinsic = pbatch["reward"][:, :T].cpu().numpy()
    assert not np.array_equal(batch["reward"][:, :T].cpu().numpy(), extrinsic)
    A = runner.env.n_actions
    per_env = []
    for b in range(B):
        env = REGISTRY["cleanup"](**runner.args.env_args, quiet=True, env_gid_base=b)
        env.reset()
        terminated, t = False, 0
        while not terminated:
            r, terminated, info = env.step((table[b:b + 1, t] % A)[0])
            assert np.array_equal(np.asarray(r, np.float32), batch["reward"][b, t].cpu().numpy()), (b, t)
            t += 1
        per_env.append(info["shaped_return"])
        assert info["collective_return"] == runner.last_env_info["collective_return"][b]
        env.close()
    per_env = np.array(per_env)
    np.testing.assert_allclose(per_env, runner.last_env_info["shaped_return"], rtol=1e-12, atol=0)
    assert logged["test_shaped_return_mean"] == pytest.approx(per_env.mean(), rel=1e-12)
    vid = runner.last_env_info["variant"]
    for v in range(2):
        assert logged[f"test_v{v}_shaped_return_mean"] == pytest.approx(per_env[vid == v].mean(), rel=1e-12)
    # without ind_reward the batch holds the agents' summed shaped reward
    summed = make_runner("cleanup", "default3", n, 7, B=B, T=T, extra=dict(obs_color="full", reward_shaping=HUGHES,
                                                                         variants=variants))
    summed.args.ind_reward = False
    e2 = summed.env
    scheme = dict(_scheme(n, A, e2.H, e2.W, e2.N), reward={"shape": (1,)})
    summed.use_batch_factory(lambda: FakeBatch(scheme, B, T + 1, e2.device))
    summed.mac = ScriptedMAC(table, table_inc)
    b2 = summed.run(test_mode=True)
    np.testing.assert_allclose(b2["reward"][:, :T, 0].cpu().numpy(), batch["reward"][:, :T].sum(-1).cpu().numpy(), rtol=1e-6)


def test_facade_returns_the_shaped_rewards():
    """The facade's step() returns the shaped per-agent rewards of the restatement applied to the extrinsic rewards a facade
    without shaping returns; info stays extrinsic and gains shaped_return."""
    from homophily_marl_b200 import REGISTRY
    base = dict(num_agents=3, map="default3", episode_limit=6, quiet=True)
    plain = REGISTRY["cleanup"](**base, extra_args=dict(disable_fire_action=False))
    shaped = REGISTRY["cleanup"](**base, extra_args=dict(disable_fire_action=False, reward_shaping=HUGHES, episode_stats=True))
    ref = ShapingRef(1, 3, shaped.sim.shaping_params)
    rs = np.random.RandomState(11)
    for ep in range(2):
        plain.reset()
        shaped.reset()
        ref.reset()
        ret = np.zeros(3, np.float32)
        for t in range(6):
            acts = [int(x) for x in rs.randint(0, plain.n_actions, size=3)]
            r0, term0, info0 = plain.step(acts)
            r1, term1, info1 = shaped.step(acts)
            ref.step(np.asarray(r0, np.int64)[None].astype(np.int8))
            assert isinstance(r1, np.ndarray) and r1.dtype == np.float64 and term0 == term1
            assert np.array_equal(np.asarray(r1, np.float32), ref.shaped[0]), (ep, t)
            ret += ref.shaped[0]
        assert term1
        assert info1["collective_return"] == info0["collective_return"] and info1["equality_metric"] == info0["equality_metric"]
        assert info1["shaped_return"] == pytest.approx(float(ret.astype(np.float64).mean()), rel=1e-12)
        assert set(info1) - set(info0) == {"shaped_return", "efficiency", "sustainability", "peace", "apples", "fires", "hits",
                                           "cleaned"}
    plain.close()
    shaped.close()


NODES = [f"tests/test_gpu_shaping.py::{t}" for t in (
    "test_shaped_rewards_match_the_restatement[0-cleanup10_full]", "test_shaped_rewards_match_the_restatement[3-cleanup10_full]",
    "test_shaped_rewards_match_the_restatement[0-harvest5]", "test_shaped_rewards_match_the_restatement[3-harvest5]",
    "test_shaped_rewards_match_the_restatement[3-harvest10_full]",
    "test_shaping_changes_no_other_byte[True-True-index4-index4]", "test_shaping_changes_no_other_byte[False-False-rgb-rgb]",
    "test_sweep_of_8_parameter_sets_equals_single_parameter_handles", "test_ranges_on_eight_streams",
    "test_autoreset_writes_the_finished_step_then_zeroes_the_trace", "test_runtime_geometry_and_custom_map")]


def test_checked_build_sees_no_shared_memory_violation():
    """The checked library (-DSSD_BOUNDS_CHECK) runs the shaping workloads of every mode, geometry, format, tagging and variant
    setting above with no shared-memory index violation (the conftest session fixture asserts the count is 0)."""
    import os
    import subprocess
    import sys
    from homophily_marl_b200 import _build
    _build.build_checked()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "-p", "no:cacheprovider", "-q", "-rA", "-m", "gpu"] + NODES, cwd=root,
                       env={**os.environ, "SSD_B200_CHECKED": "1"}, capture_output=True, text=True, timeout=3600)
    print(r.stdout[-20000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    passed = [line.split()[1] for line in r.stdout.splitlines() if line.startswith("PASSED ")]
    for node in NODES:
        assert any(p == node or p.startswith(node + "[") for p in passed), node
