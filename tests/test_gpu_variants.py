"""GPU suite: per-env variants of one handle (ssd_set_variants / ssd_set_env_variants), bit for bit.

The contract: env b running variant v equals env b of a handle created with v's config alone (same seed and env_gid_base), in
every buffer and pad byte.  A mixed batch is stepped next to one such twin handle per variant with the same inputs, and the envs
of each variant are compared with the same envs of its twin: edited layouts (walls, resources and spawn points moved), spawn
dynamics, FIRE costs and tagging-out, every shipped geometry, both colour schemes, all four (obs, state) formats, plain steps
with masked resets and auto-reset.  Also: injected draws against the C oracle built from a variant's MapSpec, env ranges on
streams with and without programmatic dependent launch, 65 536 envs, runtime geometry and a custom-size map, changing ids, a
CUDA graph, step_host, the batched runner and the validation of ssd_set_variants."""
import numpy as np
import pytest

import lockstep
from harness import (BUFS, COMBOS, END_BUFS, FIRE, ScriptedMAC, action_tables, assert_outputs_match_oracle, assert_same_buffers,
                     assert_state_matches_oracle, env_var, make_env, make_ref, make_runner, random_actions, step_one_outputs)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def edit_layout(rows, kind, seed):
    """The layout with a few interior walls added, about half the spawn points moved and some resources moved."""
    rs = np.random.RandomState(seed)
    g = [list(r) for r in rows]
    H, W = len(g), len(g[0])
    cells = lambda ch: [(r, c) for r in range(1, H - 1) for c in range(1, W - 1) if g[r][c] == ch]  # noqa: E731

    def move(ch, k):
        src = cells(ch)
        for i in rs.permutation(len(src))[:k]:
            g[src[i][0]][src[i][1]] = " "
        free = cells(" ")
        for i in rs.permutation(len(free))[:k]:
            g[free[i][0]][free[i][1]] = ch

    move("P", max(1, len(cells("P")) // 2))
    free = cells(" ")
    for i in rs.permutation(len(free))[:3]:
        g[free[i][0]][free[i][1]] = "@"
    if kind == "harvest":
        move("A", 6)
    else:
        move("B", 4)
        src = cells("H")                                     # fewer waste points: the LUTs get shorter
        for i in rs.permutation(len(src))[:2]:
            g[src[i][0]][src[i][1]] = "R"
    return ["".join(r) for r in g]


def variant_list(key):
    """Five variants: the base, other spawn dynamics, an edited layout with other costs, tagging, an edited layout with tagging."""
    from homophily_marl_b200 import mapspec
    name, mp, n, view, color = lockstep.CONFIGS[key]
    rows = mapspec.ascii_map(mapspec.params_for(name, mp).map_key)
    if name == "harvest":
        dyn = [{"spawn_prob": [0.0, 0.05, 0.08, 0.1]}, {"spawn_prob": [0.01, 0.02, 0.3, 0.5]}]
    else:
        dyn = [{"threshold_depletion": 0.6, "threshold_restoration": 0.1, "waste_spawn_prob": 0.8, "apple_respawn_prob": 0.4},
               {"apple_respawn_prob": 0.9, "waste_spawn_prob": 0.2}]
    return [{}, dyn[0],
            {"rows": edit_layout(rows, name, 1), "fire_cost": 2, "hit_penalty": 1},
            dict(dyn[1], tag_timeout=3, hit_penalty=2),
            {"rows": edit_layout(rows, name, 2), "tag_timeout": 5, "fire_cost": 0}]


def twins_of(mixed, key, **kw):
    """The single-config twin of each variant of ``mixed``."""
    return [make_env(key, mixed.B, spec=s, obs=mixed.obs_format, state=mixed.state_format, color=mixed.spec.obs_color,
                 seed=mixed.seed, limit=mixed.episode_limit, env_gid_base=mixed.env_gid_base,
                 keep_episode_end=mixed.keep_episode_end, **kw) for s in mixed.variant_specs]


def assert_like_twins(mixed, twins, what, envs=None, vid=None, bufs=None):
    """Every buffer row of the envs of each variant equals the same rows of that variant's twin."""
    vid = np.minimum(mixed.variant.cpu().numpy(), len(twins) - 1) if vid is None else vid
    envs = np.arange(mixed.B) if envs is None else np.asarray(envs)
    bufs = bufs or BUFS + (END_BUFS if mixed.keep_episode_end else ())
    got = {k: getattr(mixed, k).cpu().numpy() for k in bufs}
    for v, tw in enumerate(twins):
        m = envs[vid[envs] == v]
        if len(m) == 0:
            continue
        for k in bufs:
            want = getattr(tw, k).cpu().numpy()
            if not np.array_equal(got[k][m], want[m]):
                bad = np.argwhere(got[k][m] != want[m])[0]
                raise AssertionError((what, "variant", v, k, "env", int(m[bad[0]]), bad.tolist()))


def play(rs, env):
    """This suite's random actions (FIRE 25 %, CLEAN 15 %) on the env's device."""
    return torch.as_tensor(random_actions(rs, env, fire=0.25, clean=0.15), device=env.device)


def lockstep_all(envs, act, mode, draws=None):
    for e in envs:
        if e.keep_episode_end:
            e.end_obs_buf.fill_(0xEE)
            e.end_ep_ret_buf.fill_(-7)
            if e.end_state_buf is not None:
                e.end_state_buf.fill_(0xEE)
        if mode == "autoreset":
            e.step(act, draws=draws, want_state=True, auto_reset=True)
        else:
            e.step(act, draws=draws, want_state=True)
            done = e.done.clone()
            e.reset(mask=done, draws=draws)
            e.render(want_obs=True, want_state=True)


@pytest.mark.parametrize("mode", ["step", "autoreset"])
@pytest.mark.parametrize("key", ["harvest5", "harvest10_full", "cleanup3", "cleanup5", "cleanup10"])
def test_mixed_batch_equals_single_config_twins(key, mode):
    """Two colour schemes (the config's and the other), four format combinations, >= 2 episodes on staggered clocks."""
    B, L = 20, 9
    other = "full" if lockstep.CONFIGS[key][4] == "simplified" else "simplified"
    for i, (obs, state) in enumerate(COMBOS):
        color = lockstep.CONFIGS[key][4] if i % 2 == 0 else other
        mixed = make_env(key, B, variants=variant_list(key), obs=obs, state=state, color=color, limit=L,
                         keep_episode_end=mode == "autoreset")
        twins = twins_of(mixed, key)
        rs = np.random.RandomState(B + i)
        for e in [mixed] + twins:
            e.reset()
            e.load_state(t=np.arange(B, dtype=np.int32) % L)
        assert_like_twins(mixed, twins, (key, mode, obs, state, "reset"))
        tags = 0
        for t in range(2 * L + 2):
            lockstep_all([mixed] + twins, play(rs, mixed), mode)
            assert_like_twins(mixed, twins, (key, mode, obs, state, t))
            tags += int((mixed.tag_out > 0).sum())
        assert tags > 0                                         # the tagging variants did tag
        for e in [mixed] + twins:
            e.close()


@pytest.mark.parametrize("key", ["harvest5", "cleanup5"])
def test_tag_timeout_zero_in_a_tagging_launch_equals_the_plain_kernel(key):
    """Variants 0-2 never tag: inside launches that use the tagging kernels they equal handles without tagging."""
    B = 24
    mixed = make_env(key, B, variants=variant_list(key))
    twins = twins_of(mixed, key)
    assert [tw.spec.tag_timeout for tw in twins[:3]] == [0, 0, 0]
    rs = np.random.RandomState(5)
    for e in [mixed] + twins:
        e.reset()
    for t in range(40):
        lockstep_all([mixed] + twins, play(rs, mixed), "step")
        assert_like_twins(mixed, twins, (key, t))
    vid = mixed.variant.cpu().numpy()
    assert (mixed.tag_out.cpu().numpy()[vid < 3] == 0).all()
    assert (mixed.tag_out.cpu().numpy()[vid >= 3] > 0).any()


@pytest.mark.parametrize("key,v", [("harvest5", 4), ("harvest10_full", 2), ("cleanup5", 4), ("cleanup10", 1), ("cleanup3", 2)])
def test_injected_draws_and_teleports_against_the_oracle_of_the_variant(key, v):
    mixed = make_env(key, 1, variants=variant_list(key), variant_of=[v])
    spec = mixed.variant_specs[v]
    n = spec.n_agents
    ora = make_ref(mixed, spec=spec, seed=0)
    sched = lockstep.Schedule(70 + v, n, spec.H, spec.W, spec.n_actions, spec.wall, spec.apple_pts, spec.waste_pts,
                              spec.base_grid, teleport_every=7)
    rs = np.random.RandomState(v)
    d0 = sched.reset_draws()
    mixed.reset(draws=dict(spawn_key=d0["spawn_key"].reshape(1, n, -1), rot=d0["rot"].reshape(1, n)))
    ora.reset_one(0, dict(spawn_key=d0["spawn_key"].reshape(n, -1), rot=d0["rot"]))
    for t in range(80):
        actions, draws, tele = sched.step_inputs(t)
        actions = np.where(rs.rand(n) < 0.3, FIRE, actions).astype(np.uint8)
        rd = sched.reset_draws()
        draws.update(spawn_key=rd["spawn_key"], rot=rd["rot"])
        if tele is not None:
            mixed.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
            ora.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
        mixed.step(torch.as_tensor(actions.reshape(1, n), device=mixed.device),
                   draws={k: x.reshape(1, -1) for k, x in draws.items()}, want_state=True)
        assert_outputs_match_oracle(mixed, step_one_outputs(ora, actions, draws), (key, t))
        assert_state_matches_oracle(mixed, ora, (key, t))
        assert np.array_equal(mixed.state_rgb[0].cpu().numpy(), ora.state_one(0)), (key, t, "state")
    mixed.close()


@pytest.mark.parametrize("pdl", ["1", "0"])
@pytest.mark.parametrize("key", ["harvest5", "cleanup5"])
def test_eight_ranges_on_eight_streams_equal_one_launch(key, pdl):
    B, L, G = 8 * 40, 7, 8
    with env_var("SSD_B200_PDL", pdl):
        one, split = (make_env(key, B, variants=variant_list(key), limit=L, keep_episode_end=True) for _ in range(2))
    streams = [torch.cuda.Stream(device=one.device) for _ in range(G)]
    rs = np.random.RandomState(3)
    for e in (one, split):
        e.reset()
        e.load_state(t=np.arange(B, dtype=np.int32) % L)
    for t in range(2 * L + 1):
        act = play(rs, one)
        one.step(act, want_state=True, auto_reset=t % 2 == 0)
        main = torch.cuda.current_stream(one.device)
        for k, s in enumerate(streams):
            s.wait_stream(main)
            with torch.cuda.stream(s):
                split.step_range(act, k * (B // G), B // G, want_state=True, auto_reset=t % 2 == 0)
        for s in streams:
            main.wait_stream(s)
        assert_same_buffers(one, split, BUFS + END_BUFS, (key, pdl, t))


def test_65536_envs_sampled_and_whole_batch_invariants():
    key, B, L = "harvest5", 65536, 6
    variants = variant_list(key) + [{"spawn_prob": [0.2, 0.2, 0.2, 0.2]}, {"fire_cost": 3}, {"tag_timeout": 1}]
    mixed = make_env(key, B, variants=variants, limit=L)
    vid = mixed.variant.cpu().numpy()
    assert np.array_equal(vid, np.arange(B) % 8)
    samples = [0, 1, 7, 4097, 30001, 65534, 65535]
    twins = {b: make_env(key, 1, spec=mixed.variant_specs[vid[b]], limit=L, env_gid_base=b) for b in samples}
    rs = np.random.RandomState(1)
    mixed.reset()
    for tw in twins.values():
        tw.reset()
    for t in range(L + 2):
        act = play(rs, mixed)
        mixed.step(act, want_state=True, auto_reset=True)
        for b, tw in twins.items():
            tw.step(act[b:b + 1].contiguous(), want_state=True, auto_reset=True)
            for name in BUFS:
                assert torch.equal(getattr(mixed, name)[b:b + 1], getattr(tw, name)), (b, t, name)
        g = mixed.grid_buf[:, :mixed.G]
        counts = ((g == 2).sum(1) | ((g == 3).sum(1) << 16)).to(torch.int32)
        assert torch.equal(counts, mixed.counts_buf), t
        assert bool((mixed.t_buf == (t + 1) % L).all()), t


CUSTOM = ["@@@@@@@@@@@@@@", "@P  BB  H  RR@", "@ P BB  H  RR@", "@   @@  HS RR@", "@ BB  P  S R @", "@ BB  @  HHH @",
          "@P   BB  RR P@", "@@@@@@@@@@@@@@"]


def _runtime_case():
    from homophily_marl_b200 import mapspec
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, L = 24, 6
    base = dict(obs_color="full", random_spawn_point=True, random_spawn_rotation=None)
    variants = [{}, {"rows": edit_layout(CUSTOM, "cleanup", 3), "tag_timeout": 2},
                {"waste_spawn_prob": 0.9, "threshold_depletion": 0.5, "fire_cost": 2}]
    params = mapspec.EnvParams(mapspec.KIND_CLEANUP, "", 0.8, 0.1, 0.5, 0.3)
    mixed = SSDBatchEnv("cleanup", B, 4, view_size=4, episode_limit=L, extra_args=dict(base, variants=variants), seed=2,
                        rows=CUSTOM, params=params, want_state=True, keep_episode_end=True)
    twins = [SSDBatchEnv("cleanup", B, 4, view_size=4, episode_limit=L, extra_args=dict(base, tag_timeout=s.tag_timeout),
                         seed=2, rows=s.rows, params=s.params, fire_cost=s.fire_cost, hit_penalty=s.hit_penalty,
                         want_state=True, keep_episode_end=True) for s in mixed.variant_specs]
    rs = np.random.RandomState(0)
    for e in [mixed] + twins:
        e.reset()
    for t in range(3 * L):
        lockstep_all([mixed] + twins, play(rs, mixed), "autoreset" if t % 2 else "step")
        assert_like_twins(mixed, twins, ("custom", t))
    for key in ("harvest5", "cleanup5"):                       # shipped maps on the runtime-geometry kernels
        mixed = make_env(key, 16, variants=variant_list(key), limit=L, keep_episode_end=True)
        twins = twins_of(mixed, key)
        for e in [mixed] + twins:
            e.reset()
        for t in range(2 * L):
            lockstep_all([mixed] + twins, play(rs, mixed), "autoreset")
            assert_like_twins(mixed, twins, (key, "generic", t))


def test_custom_size_map_with_variants():
    _runtime_case()


def test_runtime_geometry_kernels():
    with env_var("SSD_B200_GENERIC", "1"):
        _runtime_case()


def test_changing_ids_then_masked_reset_equals_the_twin_of_the_new_variant():
    key, B = "cleanup5", 32
    mixed = make_env(key, B, variants=variant_list(key))
    twins = twins_of(mixed, key)
    rs = np.random.RandomState(11)
    for e in [mixed] + twins:
        e.reset()
    for t in range(5):
        lockstep_all([mixed] + twins, play(rs, mixed), "step")
    moved = np.arange(0, B, 3)
    vid = mixed.variant.cpu().numpy().astype(np.int64)
    vid[moved] = (vid[moved] + 2) % len(twins)
    vid[1] = 200                                               # past the table: runs the last variant
    mixed.variant.copy_(torch.as_tensor(vid.astype(np.uint8)))
    mask = torch.zeros(B, dtype=torch.uint8, device=mixed.device)
    mask[moved] = 1
    mask[1] = 1
    for e in [mixed] + twins:
        e.reset(mask=mask)
        e.render(want_obs=True, want_state=True)
    effective = np.minimum(vid, len(twins) - 1)
    sel = np.flatnonzero(mask.cpu().numpy())
    # a reset leaves the step outputs (reward, clean, apple_cnt, done) of the last step, taken under the old variant
    assert_like_twins(mixed, twins, "after reset", envs=sel, vid=effective, bufs=BUFS[4:])
    for t in range(20):
        lockstep_all([mixed] + twins, play(rs, mixed), "step")
        assert_like_twins(mixed, twins, ("after", t), envs=sel, vid=effective)


def test_cuda_graph_equals_eager():
    key, B, L = "harvest5", 64, 5
    eager, graphed = (make_env(key, B, variants=variant_list(key), limit=L) for _ in range(2))
    act = torch.zeros((B, eager.n), dtype=torch.uint8, device=eager.device)
    for e in (eager, graphed):
        e.reset()
    s = torch.cuda.Stream(device=eager.device)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.step(act, want_state=True, auto_reset=True)      # warm-up outside the capture
        eager.step(act, want_state=True, auto_reset=True)
        with torch.cuda.graph(g, stream=s):
            graphed.step(act, want_state=True, auto_reset=True)
    torch.cuda.current_stream().wait_stream(s)
    rs = np.random.RandomState(4)
    for t in range(3 * L):
        act.copy_(play(rs, eager))
        g.replay()
        eager.step(act, want_state=True, auto_reset=True)
        torch.cuda.synchronize()
        assert_same_buffers(eager, graphed, BUFS, t)


def test_step_host_matches_the_twins():
    key, B = "cleanup3", 12
    mixed = make_env(key, B, variants=variant_list(key))
    twins = twins_of(mixed, key)
    ios = [e.make_host_io(with_obs=True, with_state=True) for e in [mixed] + twins]
    rs = np.random.RandomState(2)
    for e in [mixed] + twins:
        e.reset()
    vid = mixed.variant.cpu().numpy()
    for t in range(15):
        act = play(rs, mixed).cpu()
        for e, io in zip([mixed] + twins, ios):
            io["actions"].copy_(act)
            e.step_host(io)
        for v in range(len(twins)):
            m = vid == v
            for k in ("reward", "clean", "apple_cnt", "done", "obs", "state"):
                assert np.array_equal(ios[0][k].numpy()[m], ios[1 + v][k].numpy()[m]), (t, v, k)


def test_batched_runner_equals_facade_runs_and_logs_per_variant():
    from homophily_marl_b200 import REGISTRY
    name, B, T = "harvest", 6, 9
    variants = [{"spawn_prob": [0, 0.005, 0.02, 0.05]}, {"spawn_prob": [0, 0.05, 0.08, 0.1], "tag_timeout": 2},
                {"fire_cost": 2}]
    logged = {}
    runner = make_runner(name, "default10", 5, 15, B=B, T=T, groups=2, extra=dict(obs_color="full", variants=variants),
                         log_stat=lambda k, v, t: logged.__setitem__(k, v))
    env_args = runner.args.env_args
    table, table_inc = action_tables(runner, 1)
    runner.mac = ScriptedMAC(table, table_inc)
    batch = runner.run(test_mode=True)
    vid = runner.last_env_info["variant"]
    assert np.array_equal(vid, np.arange(B) % 3)
    rets, colls = [], []
    for b in range(B):
        env = REGISTRY[name](**env_args, quiet=True, env_gid_base=b)
        assert int(env.sim.variant[0]) == b % 3
        env.reset()
        for t in range(T):
            st, ob = env.get_state(), np.stack(env.get_obs())
            assert np.array_equal(batch["state"][b, t].cpu().numpy(), st.astype(np.float32)), (b, t, "state")
            assert np.array_equal(batch["obs"][b, t].cpu().numpy(), ob.astype(np.float32)), (b, t, "obs")
            reward, terminated, env_info = env.step(table[b, t, :, 0])
            assert np.array_equal(batch["reward"][b, t].cpu().numpy(), reward.astype(np.float32)), (b, t, "reward")
        assert terminated
        rets.append(env.rewards.mean())
        colls.append(env_info["collective_return"])
        env.close()
    rets, colls = np.array(rets), np.array(colls)
    for k in range(3):
        m = vid == k
        assert logged[f"test_v{k}_return_mean"] == pytest.approx(rets[m].mean())
        assert logged[f"test_v{k}_collective_return_mean"] == pytest.approx(colls[m].mean())
        assert f"test_v{k}_equality_metric_mean" in logged
    assert logged["test_collective_return_mean"] == pytest.approx(colls.mean())


def test_set_variants_validation():
    from homophily_marl_b200 import _capi, mapspec
    key = "cleanup5"
    env = make_env(key, 4)
    lib, h = env.lib, env._h
    base = env.spec

    def rec(rows=None, lut=None, **kw):
        r = _capi.SsdVariant()
        a = "".join(rows or base.rows).encode()
        ta = np.ascontiguousarray(base.thr_apple if lut is None else lut, dtype=np.uint32)
        r.ascii_map, r.n_waste_lut, r.thr_apple, r.thr_waste = a, len(ta), ta.ctypes.data, ta.ctypes.data
        r.fire_cost, r.hit_penalty, r.tag_timeout = kw.get("fire_cost", 1), kw.get("hit_penalty", 0), kw.get("tag_timeout", 0)
        r._keep = (a, ta)
        return r

    def call(*recs, n=None):
        arr = (_capi.SsdVariant * max(1, len(recs)))(*recs)
        return lib.ssd_set_variants(h, len(recs) if n is None else n, arr)

    open_border = [base.rows[0][:-1] + " "] + base.rows[1:]
    bad_char = [base.rows[0]] + [base.rows[1][:3] + "x" + base.rows[1][4:]] + base.rows[2:]
    no_spawn = [r.replace("P", " ") for r in base.rows]
    assert call(rec(open_border)) == _capi.SSD_ERR_MAP
    assert call(rec(bad_char)) == _capi.SSD_ERR_MAP
    assert call(rec(), rec(no_spawn)) == _capi.SSD_ERR_SPAWN
    assert call(rec(lut=base.thr_apple[:-1])) == _capi.SSD_ERR_INVALID              # LUT length != #waste + 1
    assert call(rec(hit_penalty=30)) == _capi.SSD_ERR_INVALID                        # int8 reward bound
    assert call(rec(tag_timeout=256)) == _capi.SSD_ERR_INVALID
    assert call(rec(tag_timeout=-1)) == _capi.SSD_ERR_INVALID
    assert call(rec(), n=_capi.SSD_MAX_VARIANTS + 1) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_variants(h, -1, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_variants(h, 1, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_variants(None, 0, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_set_env_variants(None, None) == _capi.SSD_ERR_INVALID
    assert call(rec(), rec(tag_timeout=255)) == 0
    assert lib.ssd_set_variants(h, 0, None) == 0                                     # back to the creation config
    with pytest.raises(ValueError):
        make_env(key, 4, variants=[{"spawn_prob": [0, 0, 0, 0]}])
    with pytest.raises(ValueError):
        make_env(key, 4, variants=[{}, {}], variant_of=[0, 1, 2, 0])
    tagging = make_env(key, 4, variants=[{}, {"tag_timeout": 2}], variant_of=[0, 1, 0, 1])
    tagging.reset()
    with pytest.raises(ValueError, match="tag_out needs tag_timeout"):
        tagging.load_state(tag_out=np.array([[1] + [0] * 4] + [[0] * 5] * 3))
    tagging.load_state(tag_out=np.array([[0] * 5, [1] + [0] * 4, [0] * 5, [2] * 5]))
    assert mapspec.compile_variant(base, {}).thr_apple.tolist() == base.thr_apple.tolist()
    env.close()
