"""CPU suite: the reference for the per-agent episode counters (tests/stats_oracle.c, DESIGN.md §3 item 16).

The restatement steps exactly as the tagging reference (and, with tag_timeout 0, as the pinned oracle) over fuzzed steps, every
counter follows the hand-derived rules on small maps, and the four social metrics follow their definitions on hand cases."""
import numpy as np
import pytest

import lockstep
from oracle import oracle as O
from stats_oracle import (APPLE_T, APPLES, CLEANED, FIRES, HITS_DEALT, HITS_TAKEN, OUT_STEPS, StatsOracleBatch,
                          social_metrics)
from tag_oracle import TagOracleBatch

STAY, FIRE, CLEAN = 4, 7, 8
UP, DOWN, LEFT, RIGHT = 0, 1, 2, 3          # FIRE directions of orientations 0-3 (ssd_oracle.c FIRE_D)


def _spec(key):
    return lockstep.spec_for(key, episode_limit=1000)


def _fuzz_pair(key, T, B=6):
    spec = _spec(key)
    kw = dict(n_envs=B, seed=5, random_spawn_point=True, spawn_rotation=None)
    ref = TagOracleBatch.from_spec(spec, tag_timeout=T, **kw) if T else O.OracleBatch.from_spec(spec, **kw)
    return StatsOracleBatch.from_spec(spec, tag_timeout=T, **kw), ref


@pytest.mark.parametrize("key", ["cleanup5", "cleanup10_full", "harvest5", "harvest10_full"])
@pytest.mark.parametrize("T", [0, 3])
def test_restatement_steps_as_the_reference(key, T):
    """Every state and output buffer equals ssdt_step's (with tag_timeout 0 the pinned ssdo_step's): batch steps on Philox
    draws, then single-env steps with injected draws and teleports."""
    st, ref = _fuzz_pair(key, T)
    st.reset()
    ref.reset()
    rs = np.random.RandomState(1)
    n = st.n
    for t in range(40):
        a = rs.randint(0, _spec(key).n_actions, size=(st.B, n))
        a = np.where(rs.rand(st.B, n) < 0.3, FIRE, a).astype(np.uint8)
        o1, o2 = st.step(a, want_obs=True), ref.step(a, want_obs=True)
        for k in o1:
            assert np.array_equal(o1[k], o2[k]), (key, T, t, k)
        assert np.array_equal(st.envs, ref.envs), (key, T, t)
        if T:
            assert np.array_equal(st.tag_out, ref.tag_out), (key, T, t)
    sched = lockstep.schedule_for(key, 7, teleport_every=5)
    for t in range(30):
        a, d, tele = sched.step_inputs(t)
        if tele is not None:
            for o in (st, ref):
                o.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
        d = {k: v.reshape(-1) for k, v in d.items()}
        assert [np.array_equal(x, y) for x, y in zip(st.step_one(a, 0, d), ref.step_one(a, 0, d))] == [True] * 4, (key, T, t)
        assert np.array_equal(st.envs, ref.envs), (key, T, t)


def test_counters_add_up_over_fuzzed_steps():
    """Whole-batch identities: CLEANED sums clean, FIRES counts the FIRE actions (tag_timeout 0), HITS_DEALT and HITS_TAKEN total
    the same rays, APPLE_T >= APPLES, and every counter is 0 after a reset."""
    spec = _spec("cleanup5")
    st = StatsOracleBatch.from_spec(spec, n_envs=32, seed=3, random_spawn_point=True, spawn_rotation=None)
    st.reset()
    st._stats[:] = 7
    st.reset()
    assert not st.stats.any()
    rs = np.random.RandomState(2)
    clean_sum, fires = 0, 0
    for _ in range(50):
        a = rs.randint(0, spec.n_actions, size=(st.B, st.n))
        a = np.where(rs.rand(st.B, st.n) < 0.3, FIRE, a).astype(np.uint8)
        out = st.step(a, want_obs=False)
        clean_sum += out["clean"].astype(np.int64).sum()
        fires += int((a == FIRE).sum())
    s = st.stats.astype(np.int64)
    assert s[:, CLEANED].sum() == clean_sum
    assert s[:, FIRES].sum() == fires
    assert s[:, HITS_DEALT].sum() == s[:, HITS_TAKEN].sum() > 0
    assert s[:, APPLES].sum() > 0 and (s[:, APPLE_T] >= s[:, APPLES]).all()


# ---------------------------------------------------------------------------------------------------- hand-derived scenarios

ROWS = ["@@@@@@@@@",
        "@       @",
        "@       @",
        "@       @",
        "@ PPPP  @",
        "@@@@@@@@@"]


def _small(n, T=0, hit_penalty=0):
    """A 6 x 9 Cleanup map with no apple or waste points, so nothing spawns: the scenario places apples and waste itself."""
    o = StatsOracleBatch(0, ROWS, n, 3, 100, False, fire_cost=1, hit_penalty=hit_penalty, tag_timeout=T)
    o.reset_one(0)
    return o


def _place(o, cells, orient, grid=None):
    g = o.grid[0].copy() if grid is None else grid
    o.set_state(0, grid=g, pos_rc=np.array(cells), orient=np.array(orient, np.uint8))


def _grid_with(o, **cells):
    g = np.where(o.grid[0] == 1, 1, 0).astype(np.uint8)      # walls only
    for code, where in cells.items():
        for r, c in where:
            g[r, c] = {"apple": 2, "waste": 3}[code]
    return g


@pytest.mark.parametrize("hit_penalty", [0, 1])
def test_two_agents_on_one_cell_lower_eats_higher_is_hit(hit_penalty):
    """Agents 0 and 1 share an apple cell that agent 2 fires at: 0 eats, 1 takes the hit, 2 deals it -- also with
    hit_penalty 0, where no reward shows the hit."""
    o = _small(3, hit_penalty=hit_penalty)
    _place(o, [(2, 4), (2, 4), (2, 1)], [UP, UP, RIGHT], grid=_grid_with(o, apple=[(2, 4)]))
    r, _, _, _ = o.step_one(np.array([STAY, STAY, FIRE], np.uint8))
    s = o.stats[0]
    assert s[APPLES].tolist() == [1, 0, 0] and s[APPLE_T].tolist() == [1, 0, 0]
    assert s[HITS_TAKEN].tolist() == [0, 1, 0] and s[HITS_DEALT].tolist() == [0, 0, 1] and s[FIRES].tolist() == [0, 0, 1]
    assert r.tolist() == [1, -hit_penalty, -1]


def test_clean_ray_absorbed_by_an_agent_is_no_hit():
    """A CLEAN beam: the ray stopped by agent 1 hits nobody; the parallel ray cleans one waste cell."""
    o = _small(2)
    _place(o, [(2, 1), (2, 3)], [RIGHT, UP], grid=_grid_with(o, waste=[(1, 4)]))
    _, clean, _, _ = o.step_one(np.array([CLEAN, STAY], np.uint8))
    s = o.stats[0]
    assert clean.tolist() == [1, 0] and s[CLEANED].tolist() == [1, 0]
    assert not s[[FIRES, HITS_DEALT, HITS_TAKEN]].any()


def test_beam_rays_hitting_two_agents_and_two_beams_hitting_one():
    """A beam's three rays are parallel, so one beam hits an agent at most once; here its rays hit agents 1 and 2 (2 dealt),
    and agent 3's beam hits agent 2 as well (2 taken)."""
    o = _small(4)
    _place(o, [(2, 1), (1, 3), (3, 4), (3, 7)], [RIGHT, UP, UP, LEFT])
    o.step_one(np.array([FIRE, STAY, STAY, FIRE], np.uint8))
    s = o.stats[0]
    assert s[HITS_DEALT].tolist() == [2, 0, 0, 1]
    assert s[HITS_TAKEN].tolist() == [0, 1, 2, 0]
    assert s[FIRES].tolist() == [1, 0, 0, 1]


def test_tagged_agent_still_fires_and_out_steps_count_the_timeout():
    """Agents 0 and 1 fire at each other: 0 tags 1 first, 1's beam still happens and tags 0.  Both then stay out for T steps,
    which OUT_STEPS counts, and come back."""
    T = 3
    o = _small(2, T=T)
    _place(o, [(2, 1), (2, 4)], [RIGHT, LEFT])
    o.step_one(np.array([FIRE, FIRE], np.uint8))
    s = o.stats[0]
    assert s[FIRES].tolist() == [1, 1] and s[HITS_DEALT].tolist() == [1, 1] and s[HITS_TAKEN].tolist() == [1, 1]
    assert o.tag_out[0].tolist() == [T, T] and s[OUT_STEPS].tolist() == [0, 0]
    for k in range(T + 2):
        o.step_one(np.array([FIRE, FIRE], np.uint8) if k < T else np.array([STAY, STAY], np.uint8))
        assert o.stats[0][OUT_STEPS].tolist() == [min(k + 1, T)] * 2, k
    assert o.stats[0][FIRES].tolist() == [1, 1]                # actions of agents out of play are ignored


def test_apple_t_on_a_known_schedule():
    """Apples placed under agent 0 before steps 2 and 5 (and under agent 1 before step 5): APPLE_T is the sum of those t."""
    o = _small(2)
    _place(o, [(2, 2), (2, 5)], [UP, UP], grid=_grid_with(o))
    for t in range(1, 7):
        if t in (2, 5):
            cells = [(2, 2)] + ([(2, 5)] if t == 5 else [])
            o.set_state(0, grid=_grid_with(o, apple=cells))
        o.step_one(np.array([STAY, STAY], np.uint8))
    s = o.stats[0]
    assert s[APPLES].tolist() == [2, 1] and s[APPLE_T].tolist() == [7, 5]
    m = o.social_metrics()
    assert m["sustainability"][0] == pytest.approx((7 / 2 + 5 / 1) / 2, rel=1e-15)
    assert m["efficiency"][0] == pytest.approx(3 / 6, rel=1e-15)


# ---------------------------------------------------------------------------------------------------- the metric formulas

def _stats(n, **fields):
    s = np.zeros((1, 7, n), np.uint32)
    for k, v in fields.items():
        s[0, globals()[k.upper()]] = v
    return s


def test_metrics_when_no_agent_ate():
    m = social_metrics(np.array([[-2, 0, -1]]), _stats(3, fires=[2, 0, 1]), 10)
    assert m["sustainability"][0] == 0.0
    assert m["efficiency"][0] == pytest.approx(-0.3, rel=1e-15)
    assert m["peace"][0] == 3.0


def test_metrics_when_all_returns_are_zero():
    m = social_metrics(np.zeros((1, 4)), _stats(4, apples=[1, 0, 0, 1], apple_t=[3, 0, 0, 9], fires=[1, 0, 0, 1]), 8)
    assert m["efficiency"][0] == 0.0 and m["equality"][0] == 1.0   # the runners' equality_metric: 1 at a collective return of 0
    assert m["sustainability"][0] == pytest.approx(6.0, rel=1e-15)


def test_peace_with_timers_running_at_done():
    """Agents still out at the end count every step they started out of play, the ones not yet over included."""
    m = social_metrics(np.array([[4, 1, 0]]), _stats(3, out_steps=[3, 0, 2]), 10)
    assert m["peace"][0] == pytest.approx(3 - 5 / 10, rel=1e-15)
    assert m["equality"][0] == pytest.approx(1 - (2 * (3 + 4 + 1)) / (2 * 3 * 5), rel=1e-15)
