"""GPU suite: per-agent preference sets (extra_args reward_shaping as a list of one dict per agent, social value orientation,
``ssd_set_reward_preferences``; DESIGN.md §3 item 20).

After every step the shaped rewards and traces equal, bit for bit, the NumPy float32 restatement (tests/preference_ref.py) applied
to the GPU's own rewards, done flags and variant ids -- on every shipped config with and without tagging, under Philox and
injected draws, with mixed rosters and variants carrying their own, at 65 536 envs and on the runtime geometry.  A uniform
roster equals the handle without one, and svo_weight 0 equals ssd_set_reward_shaping, in every buffer; env ranges on 8 streams
(with and without programmatic dependent launch), auto-reset, masked reset, render, ssd_step_host and CUDA graphs keep the traces
right; and the batched runner's per-set statistics and the PyMARL facade's rewards follow each agent's own set."""
import ctypes as C
import math

import numpy as np
import pytest

import lockstep
from harness import (BUFS, END_BUFS, ScriptedMAC, action_tables, assert_same_buffers, env_var, make_runner, random_actions,
                     random_draws)
from preference_ref import PreferenceRef

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
HUGHES = {"alpha": 5.0, "beta": 0.05, "prosocial": 0.25}
PALETTE = [{"alpha": 5.0, "beta": 0.05}, {"prosocial": 0.5, "svo_angle": 45, "svo_weight": 0.5}, {},
           {"beta": 1.0, "svo_angle": 90, "svo_weight": 2.0, "decay": 0.9}, {"alpha": 1.0, "svo_angle": -30, "svo_weight": 0.1}]
SHAPED = ("shaped_buf", "shape_trace_buf")


def mixed(n, shift=0):
    """A mixed population: agent i takes PALETTE[(i + shift) % 5]."""
    return [PALETTE[(i + shift) % len(PALETTE)] for i in range(n)]


def make(key, B, *, shaping="mixed", obs="rgb", state="rgb", T=0, seed=9, limit=1000, **kw):
    """An SSDBatchEnv of config ``key`` (random spawn point and rotation, want_state) with reward_shaping ``shaping`` ("mixed":
    mixed(n); None: off)."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    name, mp, n, view, c = lockstep.CONFIGS[key]
    extra = dict(obs_color=c, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=T, obs_format=obs,
                 state_format=state, reward_shaping=mixed(n) if shaping == "mixed" else shaping)
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=limit, extra_args=extra, seed=seed, want_state=True, **kw)


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


def svo_active(env, ref):
    """Some agent with a non-zero svo_weight has a non-zero trace: the angle term was exercised."""
    ws = np.array([q[5] for q in env.preference_sets])
    var = np.zeros(env.B, np.int64) if env.variant is None else np.minimum(env.variant.cpu().numpy(), len(env.preference_of) - 1)
    sid = env.preference_of[var]
    return bool(((ws[sid] > 0) & (ref.trace != 0)).any())


@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
@pytest.mark.parametrize("T", [0, 3])
def test_mixed_rosters_match_the_restatement(key, T):
    env = make(key, 16, T=T, limit=30)
    n = env.n
    assert env.shaping_params is None and len(env.preference_sets) == min(n, 5)
    assert env.preference_of.tolist() == [[i % 5 for i in range(n)]]
    ref = PreferenceRef.of(env)
    env.reset()
    rs = np.random.RandomState(10 * sorted(lockstep.CONFIGS).index(key) + T)
    for t in range(40):
        at = torch.as_tensor(random_actions(rs, env, fire=0.3, clean=0.3), device=env.device)
        if t < 25:
            step_both(env, ref, at, auto_reset=t % 5 == 4)
        else:                                                 # injected draws
            step_both(env, ref, at, draws=random_draws(rs, env), want_obs=False)
        assert_matches(env, ref, (key, T, t))
    assert (env.reward != 0).any() and svo_active(env, ref)


def test_variants_with_their_own_rosters():
    """A sweep whose variants carry a list, a dict with an angle, or nothing (the handle's list): the sets are deduplicated over
    the handle and every variant, one roster row per variant."""
    n = 5
    var = [{}, {"reward_shaping": mixed(n, 2)}, {"reward_shaping": {"beta": 2.0, "svo_angle": 60, "svo_weight": 1.0}},
           {"fire_cost": 0, "reward_shaping": [{}, {}, HUGHES, HUGHES, {}]}]
    env = make("cleanup5", 256, T=3, limit=15, variants=var)
    sets = env.preference_sets
    assert len(sets) == 7 and env.preference_of.shape == (4, n)
    assert [sets[k] for k in env.preference_of[1]] == [sets[k] for k in np.roll(env.preference_of[0], -2)]
    assert len(set(env.preference_of[2].tolist())) == 1
    ref = PreferenceRef.of(env)
    env.reset()
    rs = np.random.RandomState(12)
    active, distinct = False, False
    for t in range(30):
        at = torch.as_tensor(random_actions(rs, env, fire=0.3, clean=0.3), device=env.device)
        step_both(env, ref, at, auto_reset=t % 3 == 2)
        assert_matches(env, ref, t)
        active |= svo_active(env, ref)
        vid = env.variant.cpu().numpy()
        u = env.shaped_reward().cpu().numpy()
        distinct |= len({u[vid == v].tobytes() for v in range(4)}) == 4
    assert active and distinct


@pytest.mark.parametrize("variants", [False, True])
def test_uniform_roster_and_zero_weight_equal_item_17_in_every_buffer(variants):
    """Three handles agree in every buffer over steps, ranges, auto-reset steps with episode-end buffers, masked resets, renders
    and host steps: one through ssd_set_reward_shaping; one through ssd_set_reward_preferences with an svo_angle but weight 0
    and a uniform roster (a list of identical dicts); one set directly with no roster."""
    from homophily_marl_b200 import _capi
    key, T = "harvest5", 3
    legacy = [HUGHES, {"beta": 2.0, "decay": 0.5}] if variants else [HUGHES]
    angled = [dict(q, svo_angle=30 * (k + 1)) for k, q in enumerate(legacy)]
    mk = lambda handle, own: make(key, 64, T=T, limit=12, keep_episode_end=True, shaping=handle,      # noqa: E731
                                  variants=[{}, {"reward_shaping": own}] if variants else None)
    a_env, c_env = mk(legacy[0], legacy[-1]), mk(legacy[0], legacy[-1])
    b_env = mk([angled[0]] * 5, [angled[-1]] * 5)
    assert a_env.shaping_params is not None and b_env.shaping_params is None
    assert b_env.preference_of.tolist() == a_env.preference_of.tolist()
    P = _capi.SsdPreference
    recs = (P * len(angled))(*[P(*q[:4], math.radians(15), 0.0) for q in a_env.shaping_params])
    assert c_env.lib.ssd_set_reward_preferences(c_env._h, len(recs), recs, 0, None, C.c_void_p(c_env.shape_trace_buf.data_ptr()),
                                                C.c_void_p(c_env.shaped_buf.data_ptr())) == _capi.SSD_OK
    envs = (a_env, b_env, c_env)
    rs = np.random.RandomState(4)
    t0 = rs.randint(0, 12, size=64)
    for e in envs:
        e.reset()
        e.load_state(t=t0)
    for t in range(30):
        a = random_actions(rs, a_env, fire=0.3, clean=0.2)
        at = torch.as_tensor(a, device=a_env.device)
        mode = t % 5
        for e in envs:
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
        for e in envs[1:]:
            assert_same_buffers(a_env, e, BUFS + END_BUFS + SHAPED, (variants, t))
    assert a_env.shape_trace_buf.any()


@pytest.mark.parametrize("pdl", ["1", "0"])
def test_ranges_on_eight_streams(pdl):
    """8 env ranges of 512 envs on 8 streams (with and without programmatic dependent launch) shape what one whole-batch launch
    shapes, with auto-reset steps among them."""
    var = [{}, {"reward_shaping": mixed(5, 3)}]
    with env_var("SSD_B200_PDL", pdl):
        whole, parts = make("harvest5", 4096, T=3, limit=10, variants=var), make("harvest5", 4096, T=3, limit=10, variants=var)
    streams = [torch.cuda.Stream(device=parts.device) for _ in range(8)]
    rs = np.random.RandomState(3)
    ref = PreferenceRef.of(whole)
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
        assert_same_buffers(whole, parts, BUFS + SHAPED, (pdl, t))
        assert_matches(parts, ref, (pdl, t))


def test_autoreset_masked_reset_render_and_host_step():
    """Against the restatement: auto-reset steps write the finished step and zero the traces of the envs they end, masked resets
    zero the traces they reset, ssd_render touches neither buffer, and ssd_step_host shapes as ssd_step does.  The twin without
    shaping agrees in every other buffer."""
    env = make("cleanup5", 128, T=3, limit=10, keep_episode_end=True)
    plain = make("cleanup5", 128, T=3, limit=10, keep_episode_end=True, shaping=None)
    ref = PreferenceRef.of(env)
    rs = np.random.RandomState(6)
    t0 = rs.randint(0, 10, size=128)
    for e in (env, plain):
        e.reset()
        e.load_state(t=t0)
    ended = 0
    for t in range(30):
        a = random_actions(rs, env, fire=0.4, clean=0.3)
        at = torch.as_tensor(a, device=env.device)
        mode = t % 4
        if mode == 2:
            mask = torch.as_tensor(rs.rand(128) < 0.3, device=env.device)
            u, tr = env.shaped_buf.clone(), env.shape_trace_buf.clone()
        for e in (env, plain):
            if mode == 0:
                e.step(at, auto_reset=True)
            elif mode == 1:
                e.step(at)
            elif mode == 2:
                e.reset(mask=mask)
                e.render(want_obs=True, want_state=True)
            else:
                io = e.make_host_io()
                io["actions"].copy_(torch.as_tensor(a))
                e.step_host(io)
        r, d = env.reward.cpu().numpy(), env.done.cpu().numpy()
        if mode == 0:
            ref.step(r, done=d)
            ended += int(d.sum())
            assert not env.shape_trace_buf[env.done.bool()].any()
        elif mode == 2:
            ref.reset(mask.cpu().numpy())
            assert torch.equal(env.shaped_buf, u)
            assert not env.shape_trace_buf[mask].any() and torch.equal(env.shape_trace_buf[~mask], tr[~mask])
        else:
            ref.step(r)
        assert_matches(env, ref, t)
        assert_same_buffers(env, plain, BUFS + END_BUFS, t)
    assert ended > 0 and svo_active(env, ref)


def test_cuda_graph_captured_after_the_set():
    eager, graphed = make("harvest5", 512, T=3, limit=7), make("harvest5", 512, T=3, limit=7)
    rs = np.random.RandomState(9)
    acts = [torch.as_tensor(random_actions(rs, eager, fire=0.4), device=eager.device) for _ in range(5)]
    for e in (eager, graphed):
        e.reset()
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=graphed.device)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.step(acts[0], auto_reset=True)
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
    assert_same_buffers(eager, graphed, BUFS + SHAPED, "graph")
    assert graphed.shape_trace_buf.any() and graphed.shaped_buf.any()


def test_65536_envs():
    env = make("cleanup5", 65536, limit=8, variants=[{}, {"reward_shaping": mixed(5, 1)}])
    ref = PreferenceRef.of(env)
    env.reset()
    rs = np.random.RandomState(2)
    for t in range(12):
        at = torch.as_tensor(random_actions(rs, env, fire=0.3, clean=0.3), device=env.device)
        step_both(env, ref, at, auto_reset=True, want_obs=False)
        assert_matches(env, ref, t)


def test_runtime_geometry():
    with env_var("SSD_B200_GENERIC", "1"):
        env = make("harvest5", 32, T=3, limit=12)
    ref = PreferenceRef.of(env)
    env.reset()
    rs = np.random.RandomState(8)
    for t in range(20):
        step_both(env, ref, torch.as_tensor(random_actions(rs, env, fire=0.3), device=env.device), auto_reset=t % 2 == 1)
        assert_matches(env, ref, ("generic", t))


def test_validation_on_a_live_handle():
    """Every refusal of ssd_set_reward_preferences on a real handle returns SSD_ERR_INVALID before any CUDA call and changes
    nothing; svo_angle = +-pi rounded to fp32 is accepted; n_sets = 0 with NULL, NULL turns shaping off."""
    from homophily_marl_b200 import _capi
    env = make("cleanup5", 8)
    lib, h, n = env.lib, env._h, env.n
    p = C.c_void_p(env.shaped_buf.data_ptr())
    q = C.c_void_p(env.shape_trace_buf.data_ptr())
    P = _capi.SsdPreference
    pi = float(np.float32(math.pi))
    good = (P * 2)(P(1.0, 0.5, 0.9, 0.2, pi, 1.0), P(0.0, 0.0, 1.0, 1.0, -pi, 0.0))
    roster = (C.c_uint8 * n)(*([1, 0] * n)[:n])
    over = (C.c_uint8 * n)(*([0] * (n - 1) + [2]))
    bad = [(2, good, 1, None, q, p), (2, good, 1, over, q, p), (2, None, 1, roster, q, p), (2, good, -1, roster, q, p),
           (2, good, 257, roster, q, p), (257, good, 1, roster, q, p), (-1, good, 1, roster, q, p),
           (0, None, 1, roster, None, None), (2, good, 1, roster, q, None), (2, good, 1, roster, None, p),
           (2, good, 1, roster, None, None), (0, None, 0, None, q, p), (1, good, 1, roster, q, p)]
    past = float(np.nextafter(np.float32(math.pi), np.float32(4)))
    fields = {"alpha": (math.nan, -1.0), "beta": (-0.5, math.inf), "decay": (1.5, -0.1), "prosocial": (1.01, -1.0),
              "svo_angle": (past, -past, math.nan), "svo_weight": (-0.1, math.inf)}
    for f, vals in fields.items():
        for v in vals:
            d = dict(zip([k for k, _ in P._fields_], (1.0, 0.5, 0.9, 0.2, 0.5, 1.0)))
            d[f] = v
            bad.append((1, (P * 1)(P(**d)), 0, None, q, p))
    env.reset()
    ones = torch.ones((8, n), dtype=torch.uint8, device=env.device)
    for _ in range(3):
        env.step(ones)
    torch.cuda.synchronize()
    twin = make("cleanup5", 8)
    twin.reset()
    for _ in range(3):
        twin.step(ones)
    before = lib.ssd_last_cuda_error()
    for args in bad:
        assert lib.ssd_set_reward_preferences(h, *args) == _capi.SSD_ERR_INVALID, args[:4]
    assert lib.ssd_last_cuda_error() == before
    for e in (env, twin):                                     # the handle still shapes with its own sets and roster
        e.step(ones)
    assert_same_buffers(env, twin, BUFS + SHAPED, "after refusals")
    assert lib.ssd_set_reward_preferences(h, 2, good, 1, roster, q, p) == _capi.SSD_OK          # +-pi are in range
    launches = env.launch_count
    env.step(ones)
    assert env.launch_count == launches + 2
    assert lib.ssd_set_reward_preferences(h, 0, None, 0, None, None, None) == _capi.SSD_OK
    last = env.shaped_buf.clone()
    launches = env.launch_count
    env.step(ones)
    assert env.launch_count == launches + 1 and torch.equal(env.shaped_buf, last)
    env.close()
    twin.close()


def test_batched_runner_pref_statistics_equal_facade_episodes():
    """batch["reward"] holds each agent's own shaped reward; pref{k}_return_mean and pref{k}_shaped_return_mean are the means over
    the (env, agent) pairs of set k, equal to those of the facade's episodes env for env; the extrinsic statistics equal those
    of a runner without shaping."""
    from homophily_marl_b200 import REGISTRY
    B, T, n = 6, 9, 3
    variants = [{}, {"reward_shaping": [{"beta": 3.0, "svo_angle": 45, "svo_weight": 1.0}, {}, {"prosocial": 1.0}]}]
    runs = {}
    for shaped in (False, True):
        logged = {}
        extra = dict(obs_color="full", variants=variants if shaped else [{}, {}])
        if shaped:
            extra["reward_shaping"] = [HUGHES, {"svo_angle": 90, "svo_weight": 0.5}, HUGHES]
        runner = make_runner("cleanup", "default3", n, 7, B=B, T=T, groups=1, extra=extra,
                             log_stat=lambda k, v, t, logged=logged: logged.__setitem__(k, v))
        table, table_inc = action_tables(runner, 1)
        runner.mac = ScriptedMAC(table, table_inc)
        batch = runner.run(test_mode=True)
        runs[shaped] = (runner, logged, batch)
    (plain, plog, _), (runner, logged, batch) = runs[False], runs[True]
    for k in ("test_return_mean", "test_collective_return_mean", "test_equality_metric_mean", "test_v1_return_mean"):
        assert logged[k] == plog[k], k
    assert not any(k.startswith("test_pref") for k in plog)
    e = runner.env
    assert len(e.preference_sets) == 5 and e.preference_of.tolist() == [[0, 1, 0], [2, 3, 4]]
    A = e.n_actions
    ret, sret = np.zeros((B, n)), np.zeros((B, n), np.float32)      # float32 sums in step order, as the runner's
    for b in range(B):
        env = REGISTRY["cleanup"](**runner.args.env_args, quiet=True, env_gid_base=b)
        env.reset()
        terminated, t = False, 0
        while not terminated:
            r, terminated, info = env.step((table[b:b + 1, t] % A)[0])
            assert np.array_equal(np.asarray(r, np.float32), batch["reward"][b, t].cpu().numpy()), (b, t)
            sret[b] += np.asarray(r, np.float32)
            t += 1
        ret[b] = env.rewards                                  # the facade's extrinsic episode return
        assert info["shaped_return"] == pytest.approx(sret[b].astype(np.float64).mean(), rel=1e-12)
        env.close()
    vid = runner.last_env_info["variant"]
    sid = e.preference_of[vid]
    for k in range(5):
        m = sid == k
        assert logged[f"test_pref{k}_return_mean"] == pytest.approx(ret[m].mean(), rel=1e-12), k
        assert logged[f"test_pref{k}_shaped_return_mean"] == pytest.approx(sret[m].astype(np.float64).mean(), rel=1e-12), k
    assert "test_pref5_return_mean" not in logged


def test_facade_returns_each_agents_shaped_reward():
    """The facade's step() returns the restatement's per-agent rewards for the extrinsic rewards a facade without shaping returns;
    info stays extrinsic and gains shaped_return."""
    from homophily_marl_b200 import REGISTRY
    base = dict(num_agents=3, map="default3", episode_limit=6, quiet=True)
    plain = REGISTRY["cleanup"](**base, extra_args=dict(disable_fire_action=False))
    shaped = REGISTRY["cleanup"](**base, extra_args=dict(disable_fire_action=False, reward_shaping=mixed(3, 1)))
    ref = PreferenceRef(1, 3, shaped.sim.preference_sets, set_of=shaped.sim.preference_of)
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
        assert set(info1) - set(info0) == {"shaped_return"}
    plain.close()
    shaped.close()


NODES = [f"tests/test_gpu_preferences.py::{t}" for t in (
    "test_mixed_rosters_match_the_restatement[0-cleanup10_full]", "test_mixed_rosters_match_the_restatement[3-harvest5]",
    "test_mixed_rosters_match_the_restatement[3-harvest10_full]", "test_variants_with_their_own_rosters",
    "test_uniform_roster_and_zero_weight_equal_item_17_in_every_buffer", "test_ranges_on_eight_streams",
    "test_autoreset_masked_reset_render_and_host_step", "test_runtime_geometry")]


def test_checked_build_sees_no_shared_memory_violation():
    """The checked library (-DSSD_BOUNDS_CHECK) runs the preference workloads above with no shared-memory index violation (the
    conftest session fixture asserts the count is 0)."""
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
