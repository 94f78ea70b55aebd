"""CPU suite: the NumPy restatement of the index4 state image (tests/state_index_ref.py) is pinned to the C oracle --
``color_lut[index]`` equals the oracle's RGB state image at every step of every parity configuration in both colour schemes,
with teleports (duplicate occupancy included) and with tagging-out timers -- and its layout, pack and unpack hold for odd and
even map widths."""
import numpy as np
import pytest

import lockstep
from oracle.oracle import OracleBatch
from state_index_ref import ora_state, pack, rgb_of, state_layout, unpack
from tag_oracle import TagOracleBatch

from homophily_marl_b200 import mapspec

FIRE = 7


def spec_of(key, color, **kw):
    name, mp, n, view, _ = lockstep.CONFIGS[key]
    return mapspec.compile_map(name, mp, n, view, 1000, obs_color=color, **kw)


@pytest.mark.parametrize("color", ["simplified", "full"])
@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_restatement_equals_oracle_every_step(key, color):
    spec = spec_of(key, color)
    B, full = 6, color == "full"
    ora = OracleBatch.from_spec(spec, n_envs=B, seed=11, random_spawn_point=True, spawn_rotation=None)
    ora.reset()
    rs = np.random.RandomState(len(key) + 1)
    dup = 0
    for t in range(40):
        if t % 8 == 4:                                        # teleports: clustered agents, some sharing a cell
            pos, orient = lockstep.cluster_states(rs, spec, B)
            for b in range(B):
                ora.set_state(b, pos_rc=pos[b], orient=orient[b])
                dup += len(np.unique(pos[b], axis=0)) < spec.n_agents
                assert np.array_equal(rgb_of(spec.lut, ora_state(ora, b, full)), ora.state_one(b)), (key, t, b, "cluster")
        act = rs.randint(0, spec.n_actions, size=(B, spec.n_agents)).astype(np.uint8)
        ora.step(act, want_obs=False)
        for b in range(B):
            idx = ora_state(ora, b, full)
            assert idx.max() < 16 and not (idx == 6).any()
            assert np.array_equal(rgb_of(spec.lut, idx), ora.state_one(b)), (key, t, b)
    assert dup > 0


@pytest.mark.parametrize("key", ["cleanup5", "cleanup10_full", "harvest5", "harvest10_full"])
def test_restatement_with_tagging(key):
    """tag_timeout > 0: agents out of play are absent from the state image."""
    for color in ("simplified", "full"):
        spec = spec_of(key, color, tag_timeout=3)
        B, n = 8, spec.n_agents
        ora = TagOracleBatch.from_spec(spec, n_envs=B, seed=3, random_spawn_point=True, spawn_rotation=None)
        ora.reset()
        rs = np.random.RandomState(7)
        out_seen = 0
        for t in range(40):
            a = rs.randint(0, spec.n_actions, size=(B, n))
            act = np.where(rs.rand(B, n) < 0.4, FIRE, a).astype(np.uint8)
            ora.step(act, want_obs=False)
            for b in range(B):
                tag = ora.tag_out[b]
                idx = ora_state(ora, b, color == "full", tag)
                assert np.array_equal(rgb_of(spec.lut, idx), ora.state_one(b)), (key, color, t, b)
                out_seen += int((tag > 0).sum())
        assert out_seen > 0


@pytest.mark.parametrize("H,W", [(10, 10), (25, 18), (48, 18), (9, 38), (3, 3), (7, 8), (5, 9), (12, 11), (40, 50),
                                 (32, 64), (1, 17)])
def test_layout_pack_unpack(H, W):
    rs_, env = state_layout(H, W)
    assert rs_ % 4 == 0 and rs_ >= (W + 1) // 2 and rs_ - (W + 1) // 2 < 4
    assert env % 16 == 0 and env >= H * rs_ and env - H * rs_ < 16
    assert rs_ == 4 * -(-W // 8)                              # a row is ceil(W/8) 32-bit words of 8 cells
    rng = np.random.RandomState(H * 100 + W)
    idx = rng.randint(0, 16, size=(2, H, W)).astype(np.uint8)
    buf = pack(idx)
    assert buf.shape == (2, env)
    assert np.array_equal(unpack(buf, H, W), idx)
    rows = buf[:, :H * rs_].reshape(2, H, rs_)
    c = W - 1                                                 # cell c: byte c >> 1, low nibble when c is even
    assert np.array_equal((rows[..., c >> 1] >> (4 * (c & 1))) & 15, idx[..., c])
    if W % 2:
        assert not (rows[..., W >> 1] >> 4).any()             # pad nibble of an odd width
    assert not rows[..., (W + 1) // 2:].any()                 # pad bytes of a row
    assert not buf[:, H * rs_:].any()                         # env-block tail


def test_shipped_layouts():
    """The byte counts of the shipped maps (DESIGN.md §3 item 13)."""
    assert state_layout(10, 10) == (8, 80)
    assert state_layout(25, 18) == (12, 304)
    assert state_layout(48, 18) == (12, 576)
    assert state_layout(9, 38) == (20, 192)
