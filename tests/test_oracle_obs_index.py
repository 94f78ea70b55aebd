"""CPU suite: the NumPy restatement of the index4 observations (tests/obs_index_ref.py) is pinned to the C oracle --
``color_lut[index]`` equals the oracle's RGB observation at every step of every parity configuration in both colour schemes,
with duplicate occupancy and with tagging-out timers -- and its pack / unpack helpers round-trip."""
import numpy as np
import pytest

import lockstep
from obs_index_ref import ora_index, obs_layout, pack, rgb_of, unpack
from oracle.oracle import OracleBatch
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
    rs = np.random.RandomState(len(key))
    dup = 0
    for t in range(40):
        if t % 8 == 4:                                        # clustered agents, some sharing a cell
            pos, orient = lockstep.cluster_states(rs, spec, B)
            for b in range(B):
                ora.set_state(b, pos_rc=pos[b], orient=orient[b])
                dup += len(np.unique(pos[b], axis=0)) < spec.n_agents
                assert np.array_equal(rgb_of(spec.lut, ora_index(ora, b, full)), ora.obs_one(b)), (key, t, b, "cluster")
        act = rs.randint(0, spec.n_actions, size=(B, spec.n_agents)).astype(np.uint8)
        out = ora.step(act)
        for b in range(B):
            idx = ora_index(ora, b, full)
            assert idx.max() < 16
            assert np.array_equal(rgb_of(spec.lut, idx), out["obs"][b]), (key, t, b)
    assert dup > 0


@pytest.mark.parametrize("key", ["cleanup5", "cleanup10_full", "harvest5", "harvest10_full"])
def test_restatement_with_tagging(key):
    """tag_timeout > 0: agents out of play see zeros and are absent from every other view."""
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
            out = ora.step(act)
            for b in range(B):
                tag = ora.tag_out[b]
                idx = ora_index(ora, b, color == "full", tag)
                assert not idx[tag > 0].any()
                assert np.array_equal(rgb_of(spec.lut, idx), out["obs"][b]), (key, color, t, b)
                out_seen += int((tag > 0).sum())
        assert out_seen > 0


@pytest.mark.parametrize("N", [3, 7, 11, 15, 19, 31, 63])
def test_pack_unpack_round_trip(N):
    rs = np.random.RandomState(N)
    n = 3
    idx = rs.randint(0, 16, size=(2, n, N, N)).astype(np.uint8)
    buf = pack(idx)
    rs_, agent, env = obs_layout(N, n)
    assert buf.shape == (2, env) and rs_ % 4 == 0 and rs_ >= (N + 1) // 2 and agent % 16 == 0 and agent >= N * rs_
    assert np.array_equal(unpack(buf, n, N), idx)
    rows = buf.reshape(2, n, agent)[..., :N * rs_].reshape(2, n, N, rs_)
    x = N - 1                                                 # pixel x: byte x >> 1, low nibble when x is even
    assert np.array_equal((rows[..., x >> 1] >> (4 * (x & 1))) & 15, idx[..., x])
    if N % 2:
        assert not (rows[..., N >> 1] >> 4).any()             # pad nibble
    assert not rows[..., (N + 1) // 2:].any()                 # pad bytes of a row
    assert not buf.reshape(2, n, agent)[..., N * rs_:].any()  # agent-block tail
    assert obs_layout(7 * 2 + 1, 5) == (8, 128, 640) and obs_layout(31, 5) == (16, 496, 2480)
