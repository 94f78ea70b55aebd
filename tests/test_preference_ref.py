"""CPU suite: the NumPy float32 restatement of per-agent preference sets (tests/preference_ref.py; DESIGN.md §3 item 20) on
hand-derived cases, against item 17's restatement (tests/shaping_ref.py) for a uniform roster without social value orientation,
``atan2f_ssd`` against float64 ``np.arctan2`` over the plane, and the ``reward_shaping`` keys and refusals of ``mapspec``."""
import math

import numpy as np
import pytest

from homophily_marl_b200 import mapspec
from preference_ref import ATAN_C, HALF_PI, PI, PreferenceRef, agent_sets, atan2f_ssd, f32, pref_step
from shaping_ref import DEFAULT_DECAY, shape_step


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def S(alpha=0.0, beta=0.0, decay=0.5, prosocial=0.0, svo=0.0, ws=0.0):
    return (alpha, beta, decay, prosocial, svo, ws)


# ---------------------------------------------------------------------------------------------------- atan2f_ssd

def test_coefficients_are_float32_values():
    for c in ATAN_C:
        assert float(f32(float(c))) == float(c)
    assert HALF_PI == f32(math.pi / 2) and PI == f32(math.pi)


def test_axes_diagonals_and_quadrants():
    """Exact on the axes; the diagonals and one point per quadrant are within the bound of the exact angle."""
    assert atan2f_ssd(0.0, 1.0) == 0 and atan2f_ssd(0.0, 0.0) == 0 and atan2f_ssd(-0.0, -0.0) == 0
    assert atan2f_ssd(1.0, 0.0) == HALF_PI and atan2f_ssd(-3.0, 0.0) == -HALF_PI
    assert atan2f_ssd(0.0, -2.0) == PI and atan2f_ssd(-0.0, -2.0) == PI      # signs of zero are not looked at
    for y, x in ((1, 1), (1, -1), (-1, -1), (-1, 1), (2, 5), (5, -2), (-5, -2), (-2, 5), (7, 7e-3), (-7e-3, -7)):
        assert abs(float(atan2f_ssd(y, x)) - math.atan2(y, x)) <= 2e-6, (y, x)
    assert atan2f_ssd(1.0, 1.0) == atan2f_ssd(4.0, 4.0) == atan2f_ssd(1e-40, 1e-40)          # ties |x| = |y|: q = 1


def wrapped_error(t, y, x):
    d = np.abs(t.astype(np.float64) - np.arctan2(y.astype(np.float64), x.astype(np.float64)))
    return np.minimum(d, 2 * np.pi - d)           # (+-0, x < 0) is +pi here and -pi for np.arctan2 when y = -0


def test_within_2e_6_rad_of_float64_over_the_plane():
    rs = np.random.RandomState(0)
    ang = np.linspace(-np.pi, np.pi, 1_000_001)
    pts = [(np.sin(ang), np.cos(ang))]
    for scale in (1e-42, 1e-38, 1e-3, 1.0, 37.0, 1e6, 1e30):                 # subnormals to large values
        pts.append((rs.randn(200_000) * scale, rs.randn(200_000) * scale))
    g = np.concatenate([-np.logspace(-45, 38, 300), [0.0, -0.0], np.logspace(-45, 38, 300)])
    yy, xx = np.meshgrid(g, g)
    pts.append((yy.ravel(), xx.ravel()))                                   # zeros, subnormals, ties |x| = |y| on the diagonals
    v = rs.randn(100_000).astype(f32)
    pts += [(v, v), (v, -v), (np.abs(v), v * 0)]
    y = np.concatenate([p[0] for p in pts]).astype(f32)
    x = np.concatenate([p[1] for p in pts]).astype(f32)
    both_zero = (x == 0) & (y == 0)
    t = atan2f_ssd(y, x)
    assert np.all(t[both_zero] == 0)
    err = wrapped_error(t[~both_zero], y[~both_zero], x[~both_zero])
    assert err.max() <= 2e-6, float(err.max())
    assert np.all(np.abs(t) <= PI)
    assert np.all(t[(y == 0) & (x < 0)] == PI)


def test_subnormal_inputs():
    tiny = np.array([1e-45, 3e-44, 1e-40, 1.1754942e-38], f32)
    assert tiny.min() > 0 and np.all(tiny < np.finfo(f32).tiny)
    for a in tiny:
        for b in tiny:
            assert abs(float(atan2f_ssd(a, b)) - math.atan2(float(a), float(b))) <= 2e-6, (a, b)
            assert abs(float(atan2f_ssd(-a, -b)) - math.atan2(-float(a), -float(b))) <= 2e-6, (a, b)


# ---------------------------------------------------------------------------------------------------- hand-derived steps

def test_uniform_roster_without_svo_equals_item_17():
    rs = np.random.RandomState(1)
    for n in (1, 2, 3, 5, 16):
        sets4 = [(float(rs.rand() * 5), float(rs.rand() * 5), float(rs.rand()), float(rs.rand())) for _ in range(4)]
        sets6 = [q + (float(f32(rs.rand() * 3 - 1.5)), 0.0) for q in sets4]               # an angle, but weight 0
        B = 512
        var = rs.randint(0, 6, size=B)
        r = rs.randint(-20, 20, size=(B, n)).astype(np.int8)
        trace = (rs.randn(B, n) * 30).astype(f32)
        trace[::7] = 0
        r[::5] = 0
        u17, e17 = shape_step(trace, r, sets4, var, done=var % 2)
        u, e = pref_step(trace, r, sets6, var, done=var % 2)                             # no roster: the env's set
        assert np.array_equal(bits(u), bits(u17)) and np.array_equal(bits(e), bits(e17)), n
        roster = np.repeat(np.arange(4)[:, None], n, 1)                                 # row k gives every agent set k
        u, e = pref_step(trace, r, sets6, var, set_of=roster, done=var % 2)
        assert np.array_equal(bits(u), bits(u17)) and np.array_equal(bits(e), bits(e17)), n
        u, _ = pref_step(trace, r, sets6, None, set_of=np.full((1, n), 2))
        u17, _ = shape_step(trace, r, [sets4[2]])
        assert np.array_equal(bits(u), bits(u17))


def test_a_zero_weight_subtracts_positive_zero():
    """With svo_weight 0 the angle term is +0, and u - (+0) is u bit for bit, -0 included."""
    trace, r = np.array([[0.0, 7.0, -3.0]], f32), np.array([[0, -2, 5]], np.int8)
    u, _ = pref_step(trace, r, [S(alpha=1.0, beta=2.0, svo=3.0)])
    u17, _ = shape_step(trace, r, [(1.0, 2.0, 0.5, 0.0)])
    assert np.array_equal(bits(u), bits(u17))
    z = np.array([-0.0, 0.0, -1.5], f32)
    assert np.array_equal(bits(z - f32(0)), bits(z))


def test_mixed_sets_per_agent():
    """Agent 0 is inequity-averse, agent 1 prosocial, agent 2 plain.  e = [0,0,0]*0.5 + [4, 1, 1] = [4, 1, 1]."""
    sets = [S(alpha=2.0, beta=1.0), S(prosocial=1.0), S()]
    trace, r = np.zeros((1, 3), f32), np.array([[4, 1, 1]], np.int8)
    u, e = pref_step(trace, r, sets, set_of=[[0, 1, 2]])
    assert e.tolist() == [[4, 1, 1]]
    # agent 0: D = 0, A = 3 + 3 = 6, b = 1/2: 4 - 3 = 1;  agent 1: mean reward 2;  agent 2: its own reward
    assert u.tolist() == [[1.0, 2.0, 1.0]]
    u, _ = pref_step(trace, r, sets, set_of=[[2, 1, 0]])                  # the same sets, another assignment
    assert u.tolist() == [[4.0, 2.0, 1 - 1.0 * 3]]                       # agent 2: D = 3, a = 2/2


def test_variant_rows_pick_the_roster_row_and_clamp():
    sets = [S(), S(alpha=4.0), S(prosocial=1.0)]
    roster = [[0, 0, 0], [1, 2, 0], [2, 2, 1]]
    assert agent_sets(3, 4, 3, np.array([0, 1, 2, 200]), roster).tolist() == [[0, 0, 0], [1, 2, 0], [2, 2, 1], [2, 2, 1]]
    assert agent_sets(3, 2, 3, None, roster).tolist() == [[0, 0, 0]] * 2
    assert agent_sets(3, 3, 2, np.array([0, 1, 9])).tolist() == [[0, 0], [1, 1], [2, 2]]
    trace, r = np.zeros((4, 3), f32), np.tile(np.array([[3, 0, -1]], np.int8), (4, 1))
    u, _ = pref_step(trace, r, sets, np.array([0, 1, 2, 200]), roster)
    for b, row in enumerate([0, 1, 2, 2]):
        for i in range(3):
            want, _ = pref_step(trace[b:b + 1], r[b:b + 1], [sets[roster[row][i]]])
            assert u[b, i] == want[0, i], (b, i)


def test_one_agent_has_no_angle():
    trace, r = np.array([[2.0]], f32), np.array([[3]], np.int8)
    u, e = pref_step(trace, r, [S(svo=1.0, ws=5.0)])
    assert e.tolist() == [[4.0]] and u.tolist() == [[3.0]]


def test_svo_angle_in_each_quadrant():
    """Two agents: o_0 = e_1 and th_0 = angle(e_1, e_0), so each sign pair of the traces puts th_0 in another quadrant or on
    an axis.  alpha = beta = 0 and zero rewards leave only the angle term."""
    ws, target = 2.0, float(f32(math.pi / 4))
    for e0, e1 in ((3, 1), (1, 3), (-1, 2), (-2, -5), (4, -4), (0, 0), (5, 0), (0, 5), (-5, 0), (0, -5)):
        trace, r = np.array([[e0, e1]], f32), np.zeros((1, 2), np.int8)
        u, e = pref_step(trace, r, [S(decay=1.0, svo=target, ws=ws)])
        th0, th1 = atan2f_ssd(f32(e1), f32(e0)), atan2f_ssd(f32(e0), f32(e1))
        want0 = f32(0) - f32(ws) * np.abs(f32(target) - th0)
        want1 = f32(0) - f32(ws) * np.abs(f32(target) - th1)
        assert u[0, 0] == want0 and u[0, 1] == want1, (e0, e1)
        exact = math.atan2(e1, e0) if (e0, e1) != (0, 0) else 0.0
        assert abs(float(u[0, 0]) + ws * abs(target - exact)) <= 1e-5, (e0, e1)
    # all-zero traces: the angle is 0 (individualistic), so a prosocial target costs ws * pi/4
    u, _ = pref_step(np.zeros((1, 3), f32), np.zeros((1, 3), np.int8), [S(svo=target, ws=ws)])
    assert u.tolist() == [[-float(f32(ws) * f32(target))] * 3]


def test_negative_rewards_and_others_mean():
    """Three agents, negative rewards: o_i is the plain mean of the two other traces, in ascending order."""
    trace, r = np.array([[1.0, -2.0, 0.5]], f32), np.array([[-3, 2, -1]], np.int8)
    sets = [S(decay=1.0, svo=0.0, ws=1.0)]
    u, e = pref_step(trace, r, sets)
    assert e.tolist() == [[-2.0, 0.0, -0.5]]
    o = [(f32(0.0) + f32(-0.5)) / f32(2), (f32(-2.0) + f32(-0.5)) / f32(2), (f32(-2.0) + f32(0.0)) / f32(2)]
    want = [f32(r[0, i]) - np.abs(f32(0) - atan2f_ssd(o[i], e[0, i])) for i in range(3)]
    assert u[0].tolist() == [float(x) for x in want]


def test_done_restarts_the_trace_after_writing_the_shaped_reward():
    sets = [S(alpha=1.0, svo=0.5, ws=1.0)]
    trace, r = np.array([[3, 1], [3, 1]], f32), np.array([[1, 0], [1, 0]], np.int8)
    u0, e0 = pref_step(trace, r, sets)
    u1, e1 = pref_step(trace, r, sets, done=np.array([1, 0]))
    assert np.array_equal(u0, u1) and e1[0].tolist() == [0, 0] and np.array_equal(e1[1], e0[1])


def test_reference_object_tracks_steps_resets_and_roster():
    ref = PreferenceRef(3, 2, [S(alpha=1.0), S(ws=1.0, svo=1.0)], variant=np.array([0, 1, 5]), set_of=[[0, 1], [1, 1]])
    r = np.array([[2, 0], [0, 2], [1, 1]], np.int8)
    ref.step(r)
    ref.step(r, envs=slice(0, 1))
    assert ref.trace.tolist() == [[3, 0], [0, 2], [1, 1]]
    ref.reset(np.array([0, 1, 0]))
    assert ref.trace.tolist() == [[3, 0], [0, 0], [1, 1]]
    ref.step(r, done=np.array([1, 0, 0]))
    assert ref.trace[0].tolist() == [0, 0] and ref.shaped[0, 0] == 2 - 0


# ---------------------------------------------------------------------------------------------------- mapspec keys

def test_preference_keys_and_degrees():
    assert mapspec.preference({}) == (0.0, 0.0, DEFAULT_DECAY, 0.0, 0.0, 0.0)
    q = mapspec.preference({"alpha": 5, "svo_angle": 45, "svo_weight": 0.1})
    assert q == (5.0, 0.0, DEFAULT_DECAY, 0.0, float(f32(math.radians(45))), float(f32(0.1)))
    assert mapspec.preference({"svo_angle": 180})[4] == float(PI) and mapspec.preference({"svo_angle": -180})[4] == -float(PI)
    assert mapspec.preference({"svo_angle": 90})[4] == float(HALF_PI)
    assert mapspec.reward_shaping({"alpha": 1, "svo_angle": 30}) == (1.0, 0.0, DEFAULT_DECAY, 0.0)


def test_reward_preferences_one_dict_or_one_per_agent():
    one = mapspec.reward_preferences({"beta": 2}, 3)
    assert len(one) == 3 and len(set(one)) == 1
    per = mapspec.reward_preferences([{"alpha": 1}, {}, {"svo_angle": 90, "svo_weight": 1}], 3)
    assert per[0][0] == 1.0 and per[1] == mapspec.preference({}) and per[2][4:] == (float(HALF_PI), 1.0)
    with pytest.raises(ValueError, match="one per agent"):
        mapspec.reward_preferences([{}, {}], 3)
    with pytest.raises(ValueError, match="one per agent"):
        mapspec.reward_preferences("alpha", 3)
    with pytest.raises(ValueError):
        mapspec.reward_preferences([{}, {}, 5], 3)


@pytest.mark.parametrize("bad", [{"svo_angle": 180.5}, {"svo_angle": -181}, {"svo_angle": math.nan}, {"svo_weight": -0.1},
                                 {"svo_weight": math.inf}, {"svo_weight": 1e39}, {"svo": 10}, {"svo_angle": math.inf}])
def test_preference_refuses(bad):
    with pytest.raises(ValueError):
        mapspec.preference(bad)
    with pytest.raises(ValueError):
        mapspec.reward_preferences([{}, bad], 2)


@pytest.mark.parametrize("name,mp", [("cleanup", "default3"), ("harvest", "default5")])
def test_compile_variant_takes_a_dict_or_a_list(name, mp):
    base = mapspec.compile_map(name, mp, 3, 7, 100)
    assert base.preferences is None
    sp = mapspec.compile_variant(base, {"reward_shaping": {"alpha": 5, "svo_angle": 45, "svo_weight": 0.5}})
    assert sp.preferences == (mapspec.preference({"alpha": 5, "svo_angle": 45, "svo_weight": 0.5}),) * 3
    assert sp.reward_shaping == (5.0, 0.0, DEFAULT_DECAY, 0.0)
    sp = mapspec.compile_variant(base, {"reward_shaping": [{"alpha": 5}, {}, {"prosocial": 1}], "fire_cost": 3})
    assert sp.reward_shaping is None and sp.fire_cost == 3 and sp.preferences[2][3] == 1.0
    assert mapspec.compile_variant(base, {"fire_cost": 2}).preferences is None
    with pytest.raises(ValueError):
        mapspec.compile_variant(base, {"reward_shaping": [{}, {}]})
    with pytest.raises(ValueError):
        mapspec.compile_variant(base, {"reward_shaping": [{}, {}, {"svo_angle": 200}]})


def test_batch_env_refuses_before_the_handle_exists():
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    for bad in ([{}, {}], [{}, {}, {"svo_weight": -1}], {"svo_angle": 270}, [{}, {}, {"kappa": 1}]):
        with pytest.raises(ValueError, match="reward_shaping"):
            SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(reward_shaping=bad))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            SSDBatchEnv("cleanup", 4, 3, map="default3", extra_args=dict(reward_shaping=[{}, {"svo_weight": 1}, {}]))
