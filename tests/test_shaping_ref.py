"""CPU suite: the NumPy float32 restatement of the shaped reward (tests/shaping_ref.py; DESIGN.md §3 item 17) on hand-derived
cases, against a float64 evaluation, and the ``reward_shaping`` keys of ``mapspec.compile_variant`` and ``mapspec.reward_shaping``."""
import math

import numpy as np
import pytest

from homophily_marl_b200 import mapspec
from shaping_ref import DEFAULT_DECAY, ShapingRef, f32, shape64, shape_step


def test_two_agents_with_a_known_trace():
    """e = [1, 3] * 0.5 + [2, 0] = [2.5, 1.5]: agent 0 is ahead by 1, agent 1 behind by 1."""
    trace, r = np.array([[1, 3]], f32), np.array([[2, 0]], np.int8)
    u, e = shape_step(trace, r, [(1.0, 0.5, 0.5, 0.0)])
    assert e.tolist() == [[2.5, 1.5]]
    assert u.tolist() == [[2 - 0.5 * 1, 0 - 1 * 1]]            # (r - a*D) - b*A with a = alpha, b = beta for n = 2
    u, _ = shape_step(trace, r, [(1.0, 0.5, 0.5, 0.5)])          # prosocial 0.5: m = 0.5 r + 0.5 * mean(r) = [1.5, 0.5]
    assert u.tolist() == [[1.5 - 0.5, 0.5 - 1.0]]


def test_one_agent_ignores_the_inequity_weights():
    r = np.array([[5], [-3], [0]], np.int8)
    trace = np.array([[1.5], [-2], [7]], f32)
    u, e = shape_step(trace, r, [(4.0, 9.0, 0.75, 0.3)])
    assert np.array_equal(e, trace * f32(0.75) + r.astype(f32))
    want = f32(0.7) * r.astype(f32) + f32(0.3) * (r.astype(f32) / f32(1))   # w1 = f32(1) - f32(0.3) == f32(0.7)
    assert f32(1) - f32(0.3) == f32(0.7)
    assert np.array_equal(u, want)
    u0, _ = shape_step(trace, r, [(0.0, 0.0, 0.75, 0.3)])
    assert np.array_equal(u, u0)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 16])
def test_zero_parameters_return_the_extrinsic_reward_exactly(n):
    rs = np.random.RandomState(n)
    r = rs.randint(-128, 128, size=(64, n)).astype(np.int8)
    trace = (rs.randn(64, n) * 100).astype(f32)
    for decay in (0.0, DEFAULT_DECAY, 1.0):
        u, e = shape_step(trace, r, [(0.0, 0.0, decay, 0.0)])
        assert np.array_equal(u, r.astype(f32)), decay
        assert np.array_equal(e, trace * f32(decay) + r.astype(f32))


def test_tagged_out_agent_with_zero_reward_still_counts():
    """Agent 1 is tagged out (r = 0): its trace decays and still enters the others' gaps.  e = [0, 4, 0] * 0.5 + [1, 0, 1]."""
    trace, r = np.array([[0, 4, 0]], f32), np.array([[1, 0, 1]], np.int8)
    u, e = shape_step(trace, r, [(2.0, 1.0, 0.5, 0.0)])       # a = 2/2 = 1, b = 1/2
    assert e.tolist() == [[1, 2, 1]]
    assert u.tolist() == [[1 - 1 * 1, 0 - 0.5 * 2, 1 - 1 * 1]]


def test_done_restarts_the_trace_after_writing_the_shaped_reward():
    trace, r = np.array([[3, 1], [3, 1]], f32), np.array([[1, 0], [1, 0]], np.int8)
    u0, e0 = shape_step(trace, r, [(1.0, 1.0, 1.0, 0.0)])
    u1, e1 = shape_step(trace, r, [(1.0, 1.0, 1.0, 0.0)], done=np.array([1, 0]))
    assert np.array_equal(u0, u1) and e1[0].tolist() == [0, 0] and np.array_equal(e1[1], e0[1])


def test_variant_ids_pick_the_parameter_set_and_clamp():
    params = [(0.0, 0.0, 0.5, 0.0), (5.0, 0.0, 0.5, 0.0), (0.0, 5.0, 0.5, 1.0)]
    trace, r = np.zeros((5, 3), f32), np.tile(np.array([[3, 0, -1]], np.int8), (5, 1))
    u, _ = shape_step(trace, r, params, variant=np.array([0, 1, 2, 7, 255]))
    for b, v in enumerate([0, 1, 2, 2, 2]):
        want, _ = shape_step(trace[b:b + 1], r[b:b + 1], [params[v]])
        assert np.array_equal(u[b:b + 1], want), b
    assert not np.array_equal(u[0], u[1]) and not np.array_equal(u[1], u[2])


@pytest.mark.parametrize("n", [2, 3, 5, 10, 16])
def test_restatement_equals_float64_within_float32_rounding(n):
    rs = np.random.RandomState(100 + n)
    B = 4096
    params = [(float(rs.rand() * 5), float(rs.rand() * 5), float(rs.rand()), float(rs.rand())) for _ in range(8)]
    var = rs.randint(0, 8, size=B)
    r = rs.randint(-20, 20, size=(B, n)).astype(np.int8)
    trace = (rs.randn(B, n) * 30).astype(f32)
    u, e = shape_step(trace, r, params, var)
    u64, e64 = shape64(trace, r, params, var)
    eps = 2.0 ** -24
    q = np.array(params)[var]
    assert np.all(np.abs(e - e64) <= 2 * eps * (np.abs(trace) * q[:, 2:3] + np.abs(r)))
    # every rounded operation contributes at most eps times the magnitude of its operands; (n + 6) of them touch u_i
    ea = np.abs(e64)
    gaps = ea.sum(1, keepdims=True) + n * ea
    k = 1.0 / (n - 1)
    scale = np.abs(r) + np.abs(r).mean(1, keepdims=True) + (q[:, 0:1] + q[:, 1:2]) * k * gaps
    err = np.abs(u - u64)
    assert np.all(err <= 4 * (n + 6) * eps * scale), float((err / scale).max())
    assert err.max() > 0                                      # the two evaluations do differ: float32 rounding is visible


def test_reference_object_tracks_steps_and_resets():
    ref = ShapingRef(3, 2, [(1.0, 0.0, 0.5, 0.0)])
    r = np.array([[2, 0], [0, 2], [1, 1]], np.int8)
    ref.step(r)
    ref.step(r, envs=slice(0, 1))
    assert ref.trace.tolist() == [[3, 0], [0, 2], [1, 1]]
    ref.reset(np.array([0, 1, 0]))
    assert ref.trace.tolist() == [[3, 0], [0, 0], [1, 1]]
    ref.step(r, done=np.array([1, 0, 0]))
    assert ref.trace[0].tolist() == [0, 0] and ref.shaped[0].tolist() == [2 - 0, 0 - (3.5 - 0)]


# ---------------------------------------------------------------------------------------------------- mapspec keys

def test_reward_shaping_defaults_and_float32_values():
    assert mapspec.reward_shaping({}) == (0.0, 0.0, DEFAULT_DECAY, 0.0)
    assert DEFAULT_DECAY == float(np.float32(0.99 * 0.975))
    a, b, d, w = mapspec.reward_shaping({"alpha": 0.1, "prosocial": 0.3, "decay": 1})
    assert (a, b, d, w) == (float(f32(0.1)), 0.0, 1.0, float(f32(0.3)))


@pytest.mark.parametrize("bad", [{"gamma": 0.9}, {"alpha": -1}, {"beta": -0.5}, {"decay": 1.5}, {"decay": -0.1},
                                 {"prosocial": 1.01}, {"prosocial": -1}, {"alpha": math.nan}, {"beta": math.inf}, {"alpha": 1e39}])
def test_reward_shaping_refuses(bad):
    with pytest.raises(ValueError):
        mapspec.reward_shaping(bad)


@pytest.mark.parametrize("name,mp", [("cleanup", "default3"), ("harvest", "default5")])
def test_compile_variant_reward_shaping_key(name, mp):
    base = mapspec.compile_map(name, mp, 3, 7, 100)
    assert base.reward_shaping is None
    plain = mapspec.compile_variant(base, {"fire_cost": 2})
    assert plain.reward_shaping is None and plain.fire_cost == 2   # an existing variant dict behaves as before
    sp = mapspec.compile_variant(base, {"reward_shaping": {"alpha": 5, "beta": 0.05}, "hit_penalty": 1})
    assert sp.reward_shaping == (5.0, float(f32(0.05)), DEFAULT_DECAY, 0.0) and sp.hit_penalty == 1
    assert np.array_equal(sp.base_grid, base.base_grid)
    with pytest.raises(ValueError, match="reward_shaping"):
        mapspec.compile_variant(base, {"reward_shaping": {"alpha": 1, "eta": 2}})
    with pytest.raises(ValueError):
        mapspec.compile_variant(base, {"reward_shaping": {"decay": 2}})
    assert "reward_shaping" in mapspec.VARIANT_KEYS[base.kind]
