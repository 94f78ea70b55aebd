"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the packed colour-index observations (SSD_OBS_INDEX4, DESIGN.md §3
item 12), built from an env's grid, positions, orientations and tagging-out timers.

Pixel (y, x) of agent a's view is the colour index the RGB renderer looks up: 0-5 cell codes, 6 outside the map, an agent
7 in the simplified scheme and 6 + agent_char(i) of the highest index on the cell in the full scheme (map_env.py:370).  So
``lut[index_views(...)]`` is the RGB observation.  An agent that is out of play is absent from every view and sees zeros.
"""
from __future__ import annotations

import numpy as np

from homophily_marl_b200 import mapspec

ROT_K = {mapspec.LEFT: 1, mapspec.RIGHT: 3, mapspec.UP: 0, mapspec.DOWN: 2}    # np.rot90 k (map_env.py:806-813)


def index_views(grid, pos_rc, orient, view, full, tag_out=None):
    """grid [H, W] cell codes, pos_rc [n, 2], orient [n], tag_out [n] or None -> u8 [n, N, N] colour indices."""
    grid = np.asarray(grid, dtype=np.uint8)
    pos_rc, orient = np.asarray(pos_rc), np.asarray(orient)
    n, V, N = len(pos_rc), int(view), 2 * int(view) + 1
    live = np.ones(n, bool) if tag_out is None else np.asarray(tag_out)[:n] == 0
    idx = grid.copy()
    for i in range(n):                                        # later index overwrites
        if live[i]:
            idx[pos_rc[i, 0], pos_rc[i, 1]] = mapspec.AGENT_LUT_BASE + mapspec.agent_char(i) if full else 7
    pad = np.pad(idx, V, constant_values=6)
    out = np.zeros((n, N, N), dtype=np.uint8)
    for i in range(n):
        if live[i]:
            r, c = pos_rc[i]
            out[i] = np.rot90(pad[r:r + N, c:c + N], ROT_K[int(orient[i])])
    return out


def obs_layout(N, n):
    """(row_stride, agent_stride, env_stride) of the index4 format."""
    rs = -(-((N + 1) // 2) // 4) * 4
    agent = -(-(N * rs) // 16) * 16
    return rs, agent, n * agent


def pack(idx, n_agents=None):
    """u8 [..., n, N, N] indices (< 16) -> the index4 bytes of those agent views: [..., n * agent_stride], pads zero."""
    idx = np.asarray(idx, dtype=np.uint8)
    n, N = idx.shape[-3], idx.shape[-1]
    rs, agent, _ = obs_layout(N, n)
    lead = idx.shape[:-3]
    rows = np.zeros(lead + (n, N, 2 * rs), dtype=np.uint8)
    rows[..., :N] = idx
    packed = rows[..., 0::2] | (rows[..., 1::2] << 4)                         # [..., n, N, rs]
    block = np.zeros(lead + (n, agent), dtype=np.uint8)
    block[..., :N * rs] = packed.reshape(lead + (n, N * rs))
    return block.reshape(lead + (n * agent,))


def unpack(buf, n, N):
    """Inverse of ``pack``: [..., n * agent_stride] bytes -> u8 [..., n, N, N]."""
    buf = np.asarray(buf, dtype=np.uint8)
    rs, agent, _ = obs_layout(N, n)
    lead = buf.shape[:-1]
    rows = buf.reshape(lead + (n, agent))[..., :N * rs].reshape(lead + (n, N, rs))
    both = np.stack((rows & 15, rows >> 4), axis=-1).reshape(lead + (n, N, 2 * rs))
    return both[..., :N]


def rgb_of(lut, idx):
    """u8 [..., n, N, N] indices -> u8 [..., n, 3, N, N] RGB planes (the reference's get_obs * 256)."""
    return np.moveaxis(np.asarray(lut)[idx], -1, -3)


def ora_index(ora, b, full, tag_out=None):
    """``index_views`` of env b of an ``OracleBatch`` / ``TagOracleBatch``."""
    return index_views(ora.grid[b], ora.pos_rc[b], ora.orient[b], ora.V, full, tag_out)
