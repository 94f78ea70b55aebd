"""GPU suite: per-agent episode counters (extra_args episode_stats, ``ssd_set_stats``; DESIGN.md §3 item 16).

Every counter equals the restatement in tests/stats_oracle.c after every step, on every shipped config with and without tagging,
on the runtime geometry and a custom map, at 4 096 and 65 536 envs, in env ranges on 8 streams, under auto-reset, with variants
and in CUDA graphs; a handle with counters is bit-identical to its twin without them in every other buffer; the social metrics
equal their NumPy restatement; and the batched runner and the PyMARL facade report the same metrics."""
import numpy as np
import pytest

import lockstep
from harness import (BUFS, COMBOS, CUSTOM, END_BUFS, ScriptedMAC, action_tables, assert_same_buffers,
                     assert_state_matches_oracle, custom_params, env_var, make_runner, random_actions, random_draws, random_map)
from stats_oracle import StatsOracleBatch, social_metrics

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
SOCIAL = ("efficiency", "equality", "sustainability", "peace")


def make(key, B, *, stats=True, obs="rgb", state="rgb", T=0, seed=9, limit=1000, spec=None, **kw):
    """An SSDBatchEnv of config ``key`` (random spawn point and rotation, want_state) with or without the counters; ``spec``
    supplies layout, dynamics, FIRE costs and tag_timeout instead of the config and ``T``."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    name, mp, n, view, c = lockstep.CONFIGS[key]
    extra = dict(obs_color=c, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=T if spec is None else spec.tag_timeout,
                 obs_format=obs, state_format=state, episode_stats=stats)
    if spec is not None:
        kw.update(rows=spec.rows, params=spec.params, fire_cost=spec.fire_cost, hit_penalty=spec.hit_penalty)
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=limit, extra_args=extra, seed=seed, want_state=True, **kw)


def make_oracle(env, spec=None, B=None, gid0=None):
    return StatsOracleBatch.from_spec(env.spec if spec is None else spec, n_envs=env.B if B is None else B, seed=env.seed,
                                      env_gid0=env.env_gid_base if gid0 is None else gid0,
                                      random_spawn_point=bool(env.extra_args["random_spawn_point"]),
                                      spawn_rotation=env.extra_args["random_spawn_rotation"])


def counters(env, buf=None):
    return env.stats(buf).cpu().numpy().view(np.uint32)


def assert_counters(env, ora, what, envs=slice(None)):
    got, want = counters(env)[envs], ora.stats
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError((what, "stats [env, field, agent]", bad[0].tolist(), got[tuple(bad[0])], want[tuple(bad[0])], len(bad)))


def lockstep_run(env, ora, rs, steps, fire=0.3, clean=0.3, inject=False, teleport=0):
    """Steps env and oracle with the same random actions -- Philox draws, or injected draws with teleports every ``teleport``
    steps -- and compares the counters and the state after every step."""
    for t in range(steps):
        a = random_actions(rs, env, fire=fire, clean=clean)
        at = torch.as_tensor(a, device=env.device)
        if not inject:
            env.step(at, want_obs=False)
            ora.step(a, want_obs=False, threads=8)
        else:
            if teleport and t % teleport == 0:
                pos, ori = lockstep.cluster_states(rs, env.spec, env.B)
                env.load_state(pos_rc=pos, orient=ori)
                for b in range(env.B):
                    ora.set_state(b, pos_rc=pos[b], orient=ori[b])
            d = random_draws(rs, env)
            env.step(at, draws=d, want_obs=False)
            for b in range(env.B):
                ora.step_one(a[b], b, {k: v[b].reshape(-1) for k, v in d.items()})
        assert_counters(env, ora, t)
        assert_state_matches_oracle(env, ora, t)


@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
@pytest.mark.parametrize("T", [0, 3])
def test_counters_match_the_restatement(key, T):
    env = make(key, 16, T=T)
    ora = make_oracle(env)
    env.reset()
    ora.reset()
    rs = np.random.RandomState(10 * sorted(lockstep.CONFIGS).index(key) + T)
    lockstep_run(env, ora, rs, 25)
    lockstep_run(env, ora, rs, 20, inject=True, teleport=7)
    s = counters(env)
    assert s[:, 2].sum() > 0 and s[:, 3].sum() > 0 and s[:, 0].sum() > 0          # FIREs, hits and apples happened
    if T:
        assert s[:, 5].sum() > 0
    env.close()


@pytest.mark.parametrize("obs,state", COMBOS)
@pytest.mark.parametrize("key,T", [("cleanup5", 3), ("harvest5", 3), ("cleanup10_full", 0)])
def test_counters_change_no_other_byte(key, T, obs, state):
    """A handle with counters and its twin without them agree in every buffer and pad byte over steps, ranges, auto-reset
    steps with episode-end buffers, masked resets and renders."""
    a_env = make(key, 64, T=T, obs=obs, state=state, limit=12, keep_episode_end=True)
    b_env = make(key, 64, T=T, obs=obs, state=state, limit=12, keep_episode_end=True, stats=False)
    assert b_env.stats_buf is None and b_env.end_stats_buf is None
    rs = np.random.RandomState(4)
    t0 = rs.randint(0, 12, size=64)
    for e in (a_env, b_env):
        e.reset()
        e.load_state(t=t0)
    for t in range(30):
        at = torch.as_tensor(random_actions(rs, a_env, fire=0.3, clean=0.2), device=a_env.device)
        mode = t % 4
        for e in (a_env, b_env):
            if mode == 0:
                e.step(at, want_state=True)
            elif mode == 1:
                e.step(at, want_state=True, auto_reset=True)
            elif mode == 2:
                e.step_range(at, 0, 40, want_state=True, auto_reset=True)
                e.step_range(at, 40, 24, want_state=True)
            else:
                e.reset(mask=torch.as_tensor(t0 % 3 == t % 3, device=e.device))
                e.render(want_obs=True, want_state=True)
        assert_same_buffers(a_env, b_env, BUFS + END_BUFS, (key, T, obs, state, t))
    assert counters(a_env).any()
    a_env.close()
    b_env.close()


def test_philox_batches_of_4096_and_65536_envs():
    """4 096 Harvest envs against the restatement after every step; 65 536 Cleanup envs on sampled envs (one oracle env each,
    keyed by its global id) and two whole-batch identities: CLEANED sums the episode's clean outputs and, without tagging, FIRES
    counts the FIRE actions."""
    env = make("harvest5", 4096)
    ora = make_oracle(env)
    env.reset()
    ora.reset(threads=8)
    lockstep_run(env, ora, np.random.RandomState(0), 12, fire=0.4)
    env.close()

    B = 65536
    env = make("cleanup5", B)
    sample = np.random.RandomState(1).choice(B, 24, replace=False)
    oras = [make_oracle(env, B=1, gid0=int(b)) for b in sample]
    env.reset()
    for o in oras:
        o.reset()
    rs = np.random.RandomState(2)
    clean_sum = torch.zeros((), dtype=torch.int64, device=env.device)
    fires = 0
    for t in range(15):
        a = random_actions(rs, env, fire=0.3, clean=0.3)
        env.step(torch.as_tensor(a, device=env.device), want_obs=False)
        clean_sum += env.clean.to(torch.int64).sum()
        fires += int((a == 7).sum())
        s = counters(env)
        for b, o in zip(sample, oras):
            o.step(a[b:b + 1], want_obs=False)
            assert np.array_equal(s[b], o.stats[0]), (t, int(b))
    tot = env.stats().to(torch.int64).sum((0, 2)).cpu().numpy()
    assert tot[6] == int(clean_sum) > 0 and tot[2] == fires
    env.close()


@pytest.mark.parametrize("pdl", ["1", "0"])
def test_ranges_on_eight_streams(pdl):
    """8 env ranges on 8 streams (with and without programmatic dependent launch) count what one whole-batch launch counts."""
    with env_var("SSD_B200_PDL", pdl):
        whole, parts = make("harvest5", 4096, T=3), make("harvest5", 4096, T=3)
    streams = [torch.cuda.Stream(device=parts.device) for _ in range(8)]
    rs = np.random.RandomState(3)
    for e in (whole, parts):
        e.reset()
    torch.cuda.synchronize()
    for t in range(12):
        at = torch.as_tensor(random_actions(rs, whole, fire=0.4), device=whole.device)
        whole.step(at, auto_reset=t % 3 == 2)
        main = torch.cuda.current_stream(parts.device)
        for k, s in enumerate(streams):
            s.wait_stream(main)
            with torch.cuda.stream(s):
                parts.step_range(at, 512 * k, 512, auto_reset=t % 3 == 2)
        for s in streams:
            main.wait_stream(s)
        assert_same_buffers(whole, parts, BUFS + ("stats_buf",), (pdl, t))
    assert counters(parts).any()


def test_masked_reset_zeroes_exactly_the_masked_envs():
    env = make("cleanup5", 256, T=3)
    env.reset()
    rs = np.random.RandomState(5)
    for _ in range(10):
        env.step(torch.as_tensor(random_actions(rs, env, fire=0.4, clean=0.3), device=env.device))
    before = env.stats_buf.clone()
    mask = torch.as_tensor(rs.rand(256) < 0.4, device=env.device)
    launches = env.launch_count
    env.reset(mask=mask)
    torch.cuda.synchronize()
    assert env.launch_count == launches + 2                     # the reset kernel and the counter reset
    assert not env.stats_buf[mask].any()
    assert torch.equal(env.stats_buf[~mask], before[~mask]) and before[~mask].any()
    plain = make("cleanup5", 4, stats=False)
    launches = plain.launch_count
    plain.reset()
    assert plain.launch_count == launches + 1
    # ssd_render and ssd_step_host leave the counters alone
    before = env.stats_buf.clone()
    env.render(want_obs=True, want_state=True)
    io = env.make_host_io()
    io["actions"].copy_(torch.full((256, env.n), 7, dtype=torch.uint8))
    env.step_host(io)
    assert torch.equal(env.stats_buf, before)


@pytest.mark.parametrize("key,T", [("cleanup5", 0), ("harvest5", 3)])
def test_autoreset_writes_end_stats_then_zeroes(key, T):
    """ssd_step_autoreset: end_stats of an env whose episode ended equals the counters a step-then-reset sequence shows between
    the two calls; other slots keep a sentinel; the counters are 0 after; social_metrics(end=True) equals NumPy on them."""
    fused = make(key, 128, T=T, limit=10, keep_episode_end=True)
    seq = make(key, 128, T=T, limit=10)
    rs = np.random.RandomState(6)
    t0 = rs.randint(0, 10, size=128)
    for e in (fused, seq):
        e.reset()
        e.load_state(t=t0)
    sentinel = 0x5EADBEEF
    ended_any = 0
    for t in range(25):
        at = torch.as_tensor(random_actions(rs, fused, fire=0.4, clean=0.3), device=fused.device)
        fused.end_stats_buf.fill_(sentinel)
        fused.step(at, auto_reset=True)
        seq.step(at)
        done = seq.done.bool()
        pre, pre_ret = counters(seq), seq.ep_ret.cpu().numpy()
        seq.reset(mask=done)
        d = done.cpu().numpy()
        end = fused.end_stats_buf.cpu().numpy().view(np.uint32)
        assert np.array_equal(end[d, :, :fused.n], pre[d]), t
        assert (end[~d] == sentinel).all() and (end[d, :, fused.n:] == sentinel).all(), t
        assert not counters(fused)[d].any()
        assert_same_buffers(fused, seq, ("stats_buf", "ep_ret_buf", "agent_buf", "grid_buf"), t)
        if d.any():
            ended_any += int(d.sum())
            got = {k: v.cpu().numpy()[d] for k, v in fused.social_metrics(end=True).items()}
            want = social_metrics(pre_ret[d], pre[d], fused.episode_limit)
            for k in SOCIAL:
                np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=0, err_msg=k)
    assert ended_any > 0


@pytest.mark.parametrize("key", ["harvest5", "cleanup10"])
def test_variants_equal_single_config_twins(key):
    """A batch of variants differing in fire_cost, hit_penalty and tag_timeout counts what each variant's own handle counts."""
    variants = [{}, {"fire_cost": 0, "hit_penalty": 1}, {"tag_timeout": 4, "hit_penalty": 2, "fire_cost": 2}]
    mixed = make(key, 96, variants=variants)
    twins = [make(key, 96, spec=sp) for sp in mixed.variant_specs]
    vid = mixed.variant.cpu().numpy()
    rs = np.random.RandomState(7)
    for e in [mixed] + twins:
        e.reset()
    for t in range(20):
        at = torch.as_tensor(random_actions(rs, mixed, fire=0.4, clean=0.2), device=mixed.device)
        for e in [mixed] + twins:
            e.step(at, auto_reset=t == 12)
        s = counters(mixed)
        for v, tw in enumerate(twins):
            assert np.array_equal(s[vid == v], counters(tw)[vid == v]), (t, v)
    assert counters(mixed)[:, 5].any()


def test_runtime_geometry_and_custom_map():
    with env_var("SSD_B200_GENERIC", "1"):
        env = make("cleanup5", 32, T=3)
    ora = make_oracle(env)
    env.reset()
    ora.reset()
    rs = np.random.RandomState(8)
    lockstep_run(env, ora, rs, 20)
    lockstep_run(env, ora, rs, 10, inject=True, teleport=4)
    from homophily_marl_b200.batch_env import SSDBatchEnv
    for case in (CUSTOM[0], CUSTOM[4]):
        kind, H, W, n, view, color = case
        rows = random_map(np.random.RandomState(H * W + n), kind, H, W, n_spawn=min(32, n + 3))
        extra = dict(random_spawn_point=True, random_spawn_rotation=None, obs_color=color, tag_timeout=3, episode_stats=True)
        env = SSDBatchEnv(kind, 16, n, view_size=view, episode_limit=1000, rows=rows, params=custom_params(kind), seed=9,
                          extra_args=extra, want_state=True)
        ora = make_oracle(env)
        env.reset()
        ora.reset()
        lockstep_run(env, ora, rs, 15, fire=0.4)
        env.close()


def test_cuda_graph_capture_and_replay():
    eager, graphed = make("harvest5", 512, T=3), make("harvest5", 512, T=3)
    rs = np.random.RandomState(9)
    acts = [torch.as_tensor(random_actions(rs, eager, fire=0.4), device=eager.device) for _ in range(5)]
    for e in (eager, graphed):
        e.reset()
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=graphed.device)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.step(acts[0])                                 # warm-up outside the capture, counted like any step
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for a in acts:
                graphed.step(a)
    eager.step(acts[0])
    for _ in range(3):
        g.replay()
        for a in acts:
            eager.step(a)
    torch.cuda.synchronize()
    assert_same_buffers(eager, graphed, BUFS + ("stats_buf",), "graph")
    assert counters(graphed)[:, 3].any()


def test_social_metrics_equal_numpy():
    env = make("cleanup5", 64, T=3)
    ora = make_oracle(env)
    env.reset()
    ora.reset()
    m0 = env.social_metrics()
    assert (m0["efficiency"] == 0).all() and (m0["peace"] == env.n).all() and (m0["sustainability"] == 0).all()
    lockstep_run(env, ora, np.random.RandomState(10), 30)
    got = {k: v.cpu().numpy() for k, v in env.social_metrics().items()}
    want = ora.social_metrics()
    for k in SOCIAL:
        assert got[k].dtype == np.float64 and got[k].shape == (64,)
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=0, err_msg=k)
    assert (got["sustainability"] > 0).any() and (got["peace"] < env.n).any()


RUNNER_KEYS = ("efficiency", "sustainability", "peace", "apples", "fires", "hits", "cleaned")


@pytest.mark.parametrize("groups,variants", [(1, None), (3, None), (1, [{}, {"hit_penalty": 1, "tag_timeout": 3}])])
def test_batched_runner_keys_equal_sequential_facade_episodes(groups, variants):
    from homophily_marl_b200 import REGISTRY
    B, T, n = 6, 9, 3
    logged = {}
    extra = dict(obs_color="full", episode_stats=True, tag_timeout=2)
    if variants:
        extra["variants"] = variants
    runner = make_runner("cleanup", "default3", n, 7, B=B, T=T, groups=groups, extra=extra,
                         log_stat=lambda k, v, t: logged.__setitem__(k, v))
    table, table_inc = action_tables(runner, 1)
    runner.mac = ScriptedMAC(table, table_inc)
    runner.run(test_mode=True)
    info = runner.last_env_info
    per_env = {k: [] for k in RUNNER_KEYS}
    A = runner.env.n_actions
    for b in range(B):
        env = REGISTRY["cleanup"](**runner.args.env_args, quiet=True, env_gid_base=b)
        env.reset()
        terminated, t = False, 0
        while not terminated:
            _, terminated, env_info = env.step((table[b:b + 1, t] % A)[0])
            t += 1
        for k in RUNNER_KEYS:
            per_env[k].append(env_info[k])
        assert env_info["equality_metric"] == info["equality_metric"][b]
        env.close()
    for k in RUNNER_KEYS:                                     # fp64 sums of a few terms: the same up to summation order
        np.testing.assert_allclose(np.array(per_env[k]), info[k], rtol=1e-12, atol=0, err_msg=k)
        assert logged[f"test_{k}_mean"] == pytest.approx(np.mean(per_env[k]), rel=1e-12), k
    assert max(per_env["fires"]) > 0 and min(per_env["peace"]) <= n
    if variants:
        vid = info["variant"]
        for v in range(len(variants)):
            for k in ("efficiency", "sustainability", "peace"):
                assert logged[f"test_v{v}_{k}_mean"] == pytest.approx(np.mean(np.array(per_env[k])[vid == v]), rel=1e-12)
    for k in ("collective_return", "equality_metric", "return"):
        assert f"test_{k}_mean" in logged


def test_facade_info_keys():
    from homophily_marl_b200 import REGISTRY
    base = dict(num_agents=3, map="default3", episode_limit=5, quiet=True)
    for stats in (False, True):
        env = REGISTRY["cleanup"](**base, extra_args=dict(episode_stats=stats, disable_fire_action=False))
        env.reset()
        for t in range(5):
            _, terminated, info = env.step([7, 0, 8])
        assert terminated
        want = {"collective_return", "equality_metric", "clean_num", "apple_den"} | (set(RUNNER_KEYS) if stats else set())
        assert set(info) == want, stats
        if stats:
            assert info["fires"] == 5 and info["peace"] == 3.0 and isinstance(info["efficiency"], float)
        env.close()


NODES = [f"tests/test_gpu_stats.py::{t}" for t in (
    "test_counters_match_the_restatement[0-cleanup10_full]", "test_counters_match_the_restatement[3-cleanup10_full]",
    "test_counters_match_the_restatement[0-harvest5]", "test_counters_match_the_restatement[3-harvest5]",
    "test_counters_match_the_restatement[3-harvest10_full]",
    "test_counters_change_no_other_byte[cleanup5-3-index4-index4]", "test_counters_change_no_other_byte[harvest5-3-rgb-rgb]",
    "test_counters_change_no_other_byte[harvest5-3-index4-rgb]",
    "test_autoreset_writes_end_stats_then_zeroes", "test_variants_equal_single_config_twins",
    "test_runtime_geometry_and_custom_map", "test_ranges_on_eight_streams")]


def test_checked_build_sees_no_shared_memory_violation():
    """The checked library (-DSSD_BOUNDS_CHECK) runs the counting kernels of every mode, geometry, format, tagging and variant
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
