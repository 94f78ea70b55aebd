"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of the packed colour-index state image (state_format "index4",
SSD_OBS_INDEX4 passed to ssd_set_state_format, DESIGN.md §3 item 13), built from an env's grid, positions and tagging-out
timers.

Cell (r, c) is the colour index the RGB state renderer looks up: the cell code 0-5, or where an agent in play stands the
colour index of the highest agent index on the cell (7 in the simplified scheme, 6 + agent_char(i) in the full scheme;
map_env.py:370).  So ``lut[index_state(...)]`` is the RGB state image.  An agent out of play is absent; 6 never occurs.
"""
from __future__ import annotations

import numpy as np

from homophily_marl_b200 import mapspec


def index_state(grid, pos_rc, full, tag_out=None):
    """grid [H, W] cell codes, pos_rc [n, 2], tag_out [n] or None -> u8 [H, W] colour indices."""
    idx = np.array(grid, dtype=np.uint8)
    pos_rc = np.asarray(pos_rc)
    n = len(pos_rc)
    live = np.ones(n, bool) if tag_out is None else np.asarray(tag_out)[:n] == 0
    for i in range(n):                                        # later index overwrites
        if live[i]:
            idx[pos_rc[i, 0], pos_rc[i, 1]] = mapspec.AGENT_LUT_BASE + mapspec.agent_char(i) if full else 7
    return idx


def state_layout(H, W):
    """(row_stride, env_stride) of the index4 state image."""
    rs = -(-((W + 1) // 2) // 4) * 4
    return rs, -(-(H * rs) // 16) * 16


def pack(idx):
    """u8 [..., H, W] indices (< 16) -> the index4 bytes of those state images: [..., env_stride], pads zero."""
    idx = np.asarray(idx, dtype=np.uint8)
    H, W = idx.shape[-2:]
    rs, env = state_layout(H, W)
    lead = idx.shape[:-2]
    rows = np.zeros(lead + (H, 2 * rs), dtype=np.uint8)
    rows[..., :W] = idx
    packed = rows[..., 0::2] | (rows[..., 1::2] << 4)                         # [..., H, rs]
    out = np.zeros(lead + (env,), dtype=np.uint8)
    out[..., :H * rs] = packed.reshape(lead + (H * rs,))
    return out


def unpack(buf, H, W):
    """Inverse of ``pack``: [..., env_stride] bytes -> u8 [..., H, W]."""
    buf = np.asarray(buf, dtype=np.uint8)
    rs, _ = state_layout(H, W)
    lead = buf.shape[:-1]
    rows = buf[..., :H * rs].reshape(lead + (H, rs))
    return np.stack((rows & 15, rows >> 4), axis=-1).reshape(lead + (H, 2 * rs))[..., :W]


def rgb_of(lut, idx):
    """u8 [..., H, W] indices -> u8 [..., 3, H, W] RGB planes (the reference's get_state * 256)."""
    return np.moveaxis(np.asarray(lut)[idx], -1, -3)


def ora_state(ora, b, full, tag_out=None):
    """``index_state`` of env b of an ``OracleBatch`` / ``TagOracleBatch``."""
    return index_state(ora.grid[b], ora.pos_rc[b], full, tag_out)
