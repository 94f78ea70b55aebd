"""CPU suite: the NumPy restatement of forward-offset observation windows (tests/view_offset_ref.py).

At offset 0 it equals ``obs_index_ref.index_views`` (pinned to the C oracle) on fuzzed oracle states, tagging included.  On a
small custom map it satisfies hand-derived cases in all four orientations: the agent is at pixel (V, V + f), a wall V + f cells
ahead fills the far edge x = 0, nothing behind the agent is visible at f = V, and every pixel of a view from a border or corner
cell is the map cell (or "outside") that the kernel's agent repaint maps to it.  SSDBatchEnv and the PyMARL facade refuse an
invalid view_offset before they create a handle."""
import numpy as np
import pytest

import lockstep
from obs_index_ref import index_views, ora_index
from oracle.oracle import OracleBatch
from tag_oracle import TagOracleBatch
from view_offset_ref import offset_views, rgb_buffer

from homophily_marl_b200 import mapspec

FIRE = 7


@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_offset_0_is_the_reference_view_on_fuzzed_states(key):
    name, mp, n, view, color = lockstep.CONFIGS[key]
    full = color == "full"
    for T, cls in ((0, OracleBatch), (3, TagOracleBatch)):
        spec = mapspec.compile_map(name, mp, n, view, 1000, obs_color=color, tag_timeout=T)
        ora = cls.from_spec(spec, n_envs=4, seed=5, random_spawn_point=True, spawn_rotation=None)
        ora.reset()
        rs = np.random.RandomState(len(key) + T)
        for t in range(25):
            if t % 8 == 4:
                pos, orient = lockstep.cluster_states(rs, spec, 4)
                for b in range(4):
                    ora.set_state(b, pos_rc=pos[b], orient=orient[b])
            a = rs.randint(0, spec.n_actions, size=(4, n))
            ora.step(np.where(rs.rand(4, n) < 0.3, FIRE, a).astype(np.uint8))
            for b in range(4):
                tag = ora.tag_out[b] if T else None
                got = offset_views(ora.grid[b], ora.pos_rc[b], ora.orient[b], view, 0, full, tag)
                assert np.array_equal(got, ora_index(ora, b, full, tag)), (key, T, t, b)


# ---------------------------------------------------------------------------------------------------- hand-derived cases

H = W = 15
V = 3
N = 2 * V + 1


def box(H=H, W=W):
    g = np.zeros((H, W), np.uint8)
    g[0, :] = g[-1, :] = g[:, 0] = g[:, -1] = 1               # wall
    return g


def expected_by_pixel(grid, r, c, o, f, V=V):
    """Each pixel's cell from the kernel's repaint mapping (cell -> pixel, inverted here), map cells as they are, outside 6."""
    dr, dc = (int(x) for x in mapspec.ORIENT_VEC[o])
    wr, wc = r + f * dr, c + f * dc
    N = 2 * V + 1
    out = np.zeros((N, N), np.uint8)
    for y in range(N):
        for x in range(N):
            a, b = {mapspec.UP: (y, x), mapspec.LEFT: (x, N - 1 - y), mapspec.DOWN: (N - 1 - y, N - 1 - x),
                    mapspec.RIGHT: (N - 1 - x, y)}[o]
            q, p = wr - V + a, wc - V + b
            inside = 0 <= q < grid.shape[0] and 0 <= p < grid.shape[1]
            out[y, x] = grid[q, p] if inside else 6
    return out


@pytest.mark.parametrize("o", [mapspec.LEFT, mapspec.RIGHT, mapspec.UP, mapspec.DOWN])
@pytest.mark.parametrize("f", range(V + 1))
def test_agent_at_pixel_V_V_plus_f_and_the_wall_ahead_on_the_far_edge(o, f):
    dr, dc = (int(x) for x in mapspec.ORIENT_VEC[o])
    mid = H // 2
    # the border wall the agent faces is V + f cells ahead
    r = mid if dr == 0 else (V + f if dr < 0 else H - 1 - (V + f))
    c = mid if dc == 0 else (V + f if dc < 0 else W - 1 - (V + f))
    g = box()
    view = offset_views(g, [[r, c]], [o], V, f, False)[0]
    assert view[V, V + f] == 7
    assert (view[:, 0] == 1).all()                            # the wall V + f ahead, and the wall cells beside it
    rest = view[:, 1:].copy()
    rest[V, V + f - 1] = 0
    assert set(np.unique(rest)) <= {0}                        # nothing else: empty cells only
    g7 = g.copy()
    g7[r, c] = 7
    assert np.array_equal(view, expected_by_pixel(g7, r, c, o, f))


@pytest.mark.parametrize("o", [mapspec.LEFT, mapspec.RIGHT, mapspec.UP, mapspec.DOWN])
def test_nothing_behind_is_visible_at_f_equal_V(o):
    """A second agent one cell behind the first is at pixel (V, V + f + 1) for f < V and in no pixel at f = V."""
    dr, dc = (int(x) for x in mapspec.ORIENT_VEC[o])
    r, c = H // 2, W // 2
    pos = [[r, c], [r - dr, c - dc]]
    for f in range(V + 1):
        view = offset_views(box(), pos, [o, o], V, f, True)[0]
        me, other = mapspec.AGENT_LUT_BASE + mapspec.agent_char(0), mapspec.AGENT_LUT_BASE + mapspec.agent_char(1)
        assert view[V, V + f] == me
        if f < V:
            assert view[V, V + f + 1] == other
        else:
            assert other not in view and V + f == N - 1       # the agent's own column is the last one


@pytest.mark.parametrize("f", range(V + 1))
def test_border_and_corner_agents(f):
    """Agents on every border and corner cell of the playable area, facing every way, several at once (later index on top):
    every pixel is the cell the kernel's repaint mapping gives, and cells off the map are 6."""
    rs = np.random.RandomState(f)
    g = box()
    g[rs.rand(H, W) < 0.2] = 2
    g[0, :] = g[-1, :] = g[:, 0] = g[:, -1] = 1
    cells = [(1, 1), (1, W - 2), (H - 2, 1), (H - 2, W - 2), (1, 7), (H - 2, 7), (7, 1), (7, W - 2)]
    for o in range(4):
        pos = np.array(cells)
        orient = np.full(len(cells), o)
        views = offset_views(g, pos, orient, V, f, False)
        overlay = g.copy()
        for q, p in cells:
            overlay[q, p] = 7
        for i, (q, p) in enumerate(cells):
            assert views[i][V, V + f] == 7
            assert np.array_equal(views[i], expected_by_pixel(overlay, q, p, o, f)), (o, f, (q, p))


def test_custom_geometries_match_the_pixel_mapping():
    """Odd views and non-square maps, offsets 0..V, the full colour scheme (later index on top)."""
    rs = np.random.RandomState(2)
    for Hc, Wc, Vc in ((9, 38, 15), (12, 11, 3), (20, 33, 5), (6, 5, 1)):
        g = (rs.rand(Hc, Wc) < 0.3).astype(np.uint8) * 2
        g[0, :] = g[-1, :] = g[:, 0] = g[:, -1] = 1
        free = np.argwhere(g[1:-1, 1:-1] >= 0) + 1
        n = 6
        pos = free[rs.randint(0, len(free), size=n)]
        orient = rs.randint(0, 4, size=n)
        overlay = g.copy()
        for i in range(n):
            overlay[pos[i, 0], pos[i, 1]] = mapspec.AGENT_LUT_BASE + mapspec.agent_char(i)
        for f in range(Vc + 1):
            views = offset_views(g, pos, orient, Vc, f, True)
            for i in range(n):
                assert np.array_equal(views[i], expected_by_pixel(overlay, pos[i, 0], pos[i, 1], orient[i], f, V=Vc)), (Hc, f, i)
        assert np.array_equal(offset_views(g, pos, orient, Vc, 0, True), index_views(g, pos, orient, Vc, True))


def test_tagged_out_agents_are_absent_and_see_zeros():
    g = box()
    pos, orient = [[5, 5], [5, 6], [9, 9]], [mapspec.RIGHT, mapspec.LEFT, mapspec.UP]
    views = offset_views(g, pos, orient, V, 2, False, tag_out=np.array([0, 4, 0]))
    assert not views[1].any()
    assert (views[0] == 7).sum() == 1 and views[0][V, V + 2] == 7     # agent 1 (out of play) is not drawn
    full = offset_views(g, pos, orient, V, 2, False)
    assert (full[0] == 7).sum() == 2


def test_rgb_buffer_layout():
    lut = mapspec.compile_map("cleanup", "default5", 5, 7, 100).lut
    idx = np.random.RandomState(0).randint(0, 16, size=(2, 5, 15, 15)).astype(np.uint8)
    RP, AS = 16, (3 * 15 * 16 + 15) // 16 * 16
    buf = rgb_buffer(lut, idx, RP, AS)
    assert buf.shape == (2, 5 * AS)
    planes = buf.reshape(2, 5, AS)[..., :3 * 15 * RP].reshape(2, 5, 3, 15, RP)
    assert np.array_equal(np.moveaxis(planes[..., :15], 2, -1), lut[idx])
    assert not planes[..., 15:].any() and not buf.reshape(2, 5, AS)[..., 3 * 15 * RP:].any()


# ---------------------------------------------------------------------------------------------------- refusals

@pytest.mark.parametrize("offset", [-1, 8, 100, 1.5, "2", True, None, np.float32(1)])
def test_invalid_view_offset_is_refused_before_the_handle(offset):
    from homophily_marl_b200.batch_env import SSDBatchEnv
    from homophily_marl_b200.pymarl_env import REGISTRY
    with pytest.raises(ValueError, match="view_offset"):
        SSDBatchEnv("cleanup", 4, 5, map="default5", view_size=7, extra_args=dict(view_offset=offset))
    with pytest.raises(ValueError, match="view_offset"):
        REGISTRY["cleanup"](num_agents=5, map="default5", view_size=7, quiet=True, extra_args=dict(view_offset=offset))


def test_valid_view_offsets_pass_validation():
    """0..view_size (numpy integers too) pass the check and reach the device (which this CPU machine lacks)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_gpu_view_offset.py creates these handles")
    from homophily_marl_b200.batch_env import SSDBatchEnv
    for offset in (0, 1, 7, np.int64(3)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            SSDBatchEnv("cleanup", 4, 5, map="default5", view_size=7, extra_args=dict(view_offset=offset))
