"""CPU suite: the tagging-out reference (tests/tag_oracle.c), on small hand-built maps with hand-derived expectations.

The reference is the executable form of the tagging spec (DESIGN.md §3 item 11); the GPU suite pins the kernels to it.
Orientation k fires along FIRE_D[k]: LEFT (0) up, RIGHT (1) down, UP (2) to the left, DOWN (3) to the right.  A FIRE beam
is three parallel rays: the agent's own row (or column) and the two beside it, each starting level with the agent.
"""
import numpy as np
import pytest

from homophily_marl_b200 import mapspec
from oracle.oracle import OracleBatch
from tag_oracle import TagOracleBatch

LEFT, RIGHT, UP, DOWN = 0, 1, 2, 3
STAY, CW, FIRE, CLEAN = 4, 5, 7, 8
HARVEST = ["@@@@@@@@@@@",
           "@P   P   P@",
           "@         @",
           "@         @",
           "@         @",
           "@P   A   P@",
           "@@@@@@@@@@@"]
CLEANUP = ["@@@@@@@@@@@",
           "@P   P   P@",
           "@         @",
           "@         @",
           "@         @",
           "@P       P@",
           "@@@@@@@@@@@"]
W = len(HARVEST[0])
SPAWN = [(1, 1), (1, 5), (1, 9), (5, 1), (5, 9)]      # row-major: a fixed-order respawn takes the last free one
AGENT_RGB = [(159, 67, 255), (2, 81, 154), (204, 0, 204)]   # full-colour agents 0, 1, 2


def make(T, pos, orient, tag_out=None, rows=HARVEST, hit_penalty=0, spawn_prob=(0, 0, 0, 0), random_spawn=False, view=5):
    kind = mapspec.KIND_HARVEST if rows is HARVEST else mapspec.KIND_CLEANUP
    o = TagOracleBatch(kind, rows, len(pos), view, 1000, True, spawn_prob=spawn_prob, hit_penalty=hit_penalty,
                       random_spawn_point=random_spawn, spawn_rotation=None if random_spawn else 0, tag_timeout=T)
    o.reset_one(0)
    o.set_state(0, pos_rc=np.array(pos), orient=np.array(orient, dtype=np.uint8), tag_out=tag_out)
    return o


def step(o, actions, draws=None):
    r, c, cnt, done = o.step_one(np.array(actions, dtype=np.uint8), 0, draws)
    return r.astype(int).tolist()


def shows(img, rgb):
    """Pixels of colour rgb in a [..., 3, X, Y] image."""
    img = np.asarray(img)
    return int(np.all(np.moveaxis(img, -3, -1) == np.array(rgb, dtype=np.uint8), axis=-1).sum())


def rc(o, i):
    return tuple(int(x) for x in o.pos_rc[0, i])


def test_fire_tags_the_target_for_exactly_T_steps_then_it_respawns_fixed_order():
    T = 3
    # 0 fires right along row 3 and hits 1; 1 faces left towards 0 and keeps pressing FIRE while it is out
    o = make(T, [(3, 2), (3, 5), (5, 7)], [DOWN, UP, LEFT])
    assert step(o, [FIRE, STAY, STAY]) == [-1, 0, 0]
    assert o.tag_out[0].tolist() == [0, T, 0]
    assert rc(o, 1) == (3, 5) and o.orient[0, 1] == UP            # the record keeps where it was tagged
    for k in range(T):                                             # steps t+1 .. t+T: actions (FIRE, moves) are ignored
        obs, state = o.obs_one(0), o.state_one(0)
        assert not obs[1].any()                                    # its own view is all zero
        assert shows(obs[[0, 2]], AGENT_RGB[1]) == 0 and shows(state, AGENT_RGB[1]) == 0
        assert shows(state, AGENT_RGB[0]) == 1
        assert step(o, [STAY, FIRE if k % 2 == 0 else 0, STAY]) == [0, 0, 0]
        assert o.tag_out[0, 0] == 0 and o.ep_ret[0, 1] == 0       # nobody was hit, nothing was paid
        if k < T - 1:
            assert o.tag_out[0, 1] == T - 1 - k and rc(o, 1) == (3, 5)
    assert o.tag_out[0, 1] == 0                                    # back in the observation of step t+T
    assert rc(o, 1) == (5, 9) and o.orient[0, 1] == LEFT          # last free spawn point, spawn_rotation 0
    assert shows(o.state_one(0), AGENT_RGB[1]) == 1 and o.obs_one(0)[1].any()
    o.set_state(0, orient=np.array([DOWN, UP, LEFT], dtype=np.uint8))
    o.set_state(0, pos_rc=np.array([(3, 2), (3, 5), (5, 7)]))
    assert step(o, [STAY, FIRE, STAY]) == [0, -1, 0]               # it acts again from step t+T+1
    assert o.tag_out[0].tolist() == [T, 0, 0]


def test_respawn_in_keyed_order_reads_the_injected_draws():
    o = make(2, [(3, 2), (3, 5), (5, 7)], [DOWN, UP, LEFT], random_spawn=True)
    step(o, [FIRE, STAY, STAY])
    step(o, [STAY, STAY, STAY])
    key = np.zeros((3, 7 * W), dtype=np.uint32)
    key[1, 1 * W + 5] = 7                                          # agent 1 prefers (1, 5)
    key[1, 5 * W + 1] = 7                                          # ... or (5, 1): equal keys, the larger cell wins
    draws = dict(spawn_key=key, rot=np.array([0, RIGHT, 0], dtype=np.uint8))
    step(o, [STAY, STAY, STAY], draws)
    assert o.tag_out[0, 1] == 0 and rc(o, 1) == (5, 1) and o.orient[0, 1] == RIGHT
    assert rc(o, 0) == (3, 2) and o.orient[0, 0] == DOWN          # only the respawning agent reads the draws


def test_timeout_one():
    o = make(1, [(3, 2), (3, 5), (5, 7)], [DOWN, UP, LEFT])
    step(o, [FIRE, STAY, STAY])
    assert o.tag_out[0, 1] == 1 and not o.obs_one(0)[1].any()
    assert step(o, [STAY, FIRE, STAY]) == [0, 0, 0]                # the single step out: its FIRE is ignored
    assert o.tag_out[0].tolist() == [0, 0, 0] and rc(o, 1) == (5, 9)
    assert o.obs_one(0)[1].any()


def test_a_ray_stops_at_the_first_agent():
    o = make(5, [(3, 2), (3, 4), (3, 6)], [DOWN, LEFT, LEFT])
    step(o, [FIRE, STAY, STAY])
    assert o.tag_out[0].tolist() == [0, 5, 0]


def test_a_shared_cell_tags_only_the_last_index_and_stays_occupied():
    o = make(5, [(3, 2), (3, 5), (3, 5)], [DOWN, LEFT, LEFT])
    step(o, [FIRE, STAY, STAY])
    assert o.tag_out[0].tolist() == [0, 0, 5]
    state = o.state_one(0)
    assert shows(state, AGENT_RGB[1]) == 1 and shows(state, AGENT_RGB[2]) == 0


def test_clean_never_tags_but_fire_does_in_cleanup():
    o = make(5, [(3, 2), (3, 5), (5, 7)], [DOWN, UP, LEFT], rows=CLEANUP)
    step(o, [CLEAN, STAY, STAY])
    assert o.tag_out[0].tolist() == [0, 0, 0]
    step(o, [FIRE, STAY, STAY])
    assert o.tag_out[0].tolist() == [0, 5, 0]


def test_tagged_agent_still_absorbs_later_rays_and_pays_every_hit():
    # 0 tags 1; 1 (already tagged) still fires, pays, and tags 2; 2 (already tagged) fires back and hits 1 again
    o = make(4, [(3, 2), (3, 4), (3, 6)], [DOWN, DOWN, UP], hit_penalty=2)
    assert step(o, [FIRE, FIRE, FIRE]) == [-1, -1 - 2 - 2, -1 - 2]
    assert o.tag_out[0].tolist() == [0, 4, 4]


def test_an_apple_can_spawn_under_a_just_tagged_agent():
    G = 7 * W
    draws = dict(u_apple=np.zeros(G, dtype=np.uint32))           # every eligible apple point grows (probability 1)
    o = make(3, [(5, 2), (5, 5), (1, 3)], [DOWN, UP, LEFT], spawn_prob=(1, 1, 1, 1))
    step(o, [FIRE, STAY, STAY], draws)                             # 1 stands on the apple point (5, 5) and is tagged
    assert o.tag_out[0, 1] == 3 and o.grid[0, 5, 5] == mapspec.APPLE
    ref = make(0, [(5, 2), (5, 5), (1, 3)], [DOWN, UP, LEFT], spawn_prob=(1, 1, 1, 1))
    step(ref, [FIRE, STAY, STAY], draws)                           # without tagging the agent keeps the cell empty
    assert ref.grid[0, 5, 5] == mapspec.EMPTY


def test_simultaneous_respawns_take_distinct_points_and_skip_occupied_ones():
    # 0 (in play) stands on the last spawn point; 1 and 2 come back in the same step
    o = make(5, [(5, 9), (3, 3), (3, 7)], [LEFT, LEFT, LEFT], tag_out=[0, 1, 1])
    assert step(o, [STAY, FIRE, 0]) == [0, 0, 0]
    assert o.tag_out[0].tolist() == [0, 0, 0]
    assert rc(o, 1) == (5, 1) and rc(o, 2) == (1, 9)
    # an out agent does not block a move into its cell
    o = make(5, [(3, 4), (3, 5), (1, 1)], [DOWN, LEFT, LEFT], tag_out=[0, 3, 0])
    step(o, [2, STAY, STAY])                                       # DOWN-facing action 2 moves one column right
    assert rc(o, 0) == (3, 5) and rc(o, 1) == (3, 5) and o.tag_out[0, 1] == 2


def test_reset_clears_timers():
    o = make(5, [(3, 2), (3, 5), (5, 7)], [DOWN, UP, LEFT], tag_out=[3, 0, 9])
    o.reset_one(0)
    assert o.tag_out[0].tolist() == [0, 0, 0]


@pytest.mark.parametrize("key", ["cleanup5", "harvest5", "harvest10_full"])
def test_timeout_zero_is_the_reference_trajectory(key):
    """With tag_timeout 0 the tagging reference computes what the pinned oracle computes, byte for byte."""
    from lockstep import spec_for
    spec = spec_for(key, episode_limit=40)
    B, rs = 16, np.random.RandomState(3)
    runs = [OracleBatch.from_spec(spec, n_envs=B, seed=5, random_spawn_point=True, spawn_rotation=None),
            TagOracleBatch.from_spec(spec, n_envs=B, seed=5, random_spawn_point=True, spawn_rotation=None, tag_timeout=0)]
    for o in runs:
        o.reset()
    for t in range(60):
        act = rs.randint(0, spec.n_actions, size=(B, spec.n_agents)).astype(np.uint8)
        outs = [o.step(act) for o in runs]
        for k in outs[0]:
            assert np.array_equal(outs[0][k], outs[1][k]), (t, k)
        assert runs[0].envs.tobytes() == runs[1].envs.tobytes(), t
        assert all(np.array_equal(runs[0].state_one(b), runs[1].state_one(b)) for b in range(B)), t
        if outs[0]["done"].all():
            for o in runs:
                o.reset()
    assert not runs[1].tag_out.any()


def test_tagging_fuzz_is_consistent():
    """Random FIRE-heavy play: timers stay in range, out agents get zero rewards and views, nobody stands on a wall."""
    spec = mapspec.compile_map("harvest", "default5", 5, 7, 1000, tag_timeout=4)
    B, rs = 8, np.random.RandomState(11)
    o = TagOracleBatch.from_spec(spec, n_envs=B, seed=2, random_spawn_point=True, spawn_rotation=None)
    assert o.tag_timeout == 4
    o.reset()
    seen = 0
    for t in range(200):
        act = np.where(rs.rand(B, 5) < 0.4, FIRE, rs.randint(0, 7, size=(B, 5))).astype(np.uint8)
        was_out = o.tag_out.copy()
        out = o.step(act)
        assert (out["reward"][was_out > 0] == 0).all()
        assert (out["obs"][o.tag_out > 0] == 0).all()
        assert o.tag_out.max() <= 4
        assert (np.asarray(spec.wall)[o.pos] == 0).all()
        seen += int((o.tag_out == 4).sum())
    assert seen > 20


def test_compile_map_range():
    with pytest.raises(ValueError):
        mapspec.compile_map("cleanup", "default5", 5, 7, 100, tag_timeout=256)
    with pytest.raises(ValueError):
        mapspec.compile_map("cleanup", "default5", 5, 7, 100, tag_timeout=-1)
    assert mapspec.compile_map("cleanup", "default5", 5, 7, 100).tag_timeout == 0
