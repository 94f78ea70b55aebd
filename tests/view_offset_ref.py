"""TEST INFRASTRUCTURE ONLY -- NumPy restatement of forward-offset observation windows (extra_args view_offset,
``ssd_set_view_offset``; DESIGN.md §3 item 18), built from an env's grid, positions, orientations and tagging-out timers.

The view of an agent at (r, c) facing o is ``obs_index_ref.index_views``' view with the window centred on (r + f*dr, c + f*dc),
(dr, dc) = ``mapspec.ORIENT_VEC[o]``: the map is padded by V + f cells of "outside" (index 6) instead of V, and the N x N crop
is cut around the shifted cell, then rotated by orientation as before.  f = 0 is ``index_views`` exactly.
"""
from __future__ import annotations

import numpy as np

from homophily_marl_b200 import mapspec
from obs_index_ref import ROT_K


def offset_views(grid, pos_rc, orient, view, offset, full, tag_out=None):
    """grid [H, W] cell codes, pos_rc [n, 2], orient [n], tag_out [n] or None -> u8 [n, N, N] colour indices."""
    grid = np.asarray(grid, dtype=np.uint8)
    pos_rc, orient = np.asarray(pos_rc), np.asarray(orient)
    n, V, f = len(pos_rc), int(view), int(offset)
    N = 2 * V + 1
    live = np.ones(n, bool) if tag_out is None else np.asarray(tag_out)[:n] == 0
    idx = grid.copy()
    for i in range(n):                                        # later index overwrites
        if live[i]:
            idx[pos_rc[i, 0], pos_rc[i, 1]] = mapspec.AGENT_LUT_BASE + mapspec.agent_char(i) if full else 7
    pad = np.pad(idx, V + f, constant_values=6)
    out = np.zeros((n, N, N), dtype=np.uint8)
    for i in range(n):
        if live[i]:
            o = int(orient[i])
            dr, dc = (int(x) for x in mapspec.ORIENT_VEC[o])
            r, c = pos_rc[i, 0] + f * dr + f, pos_rc[i, 1] + f * dc + f     # top-left corner of the crop in the padded map
            out[i] = np.rot90(pad[r:r + N, c:c + N], ROT_K[o])
    return out


def rgb_buffer(lut, idx, row_stride, agent_stride):
    """u8 [..., n, N, N] indices -> the RGB observation bytes [..., n * agent_stride] of those views, row and block pads zero."""
    idx = np.asarray(idx, dtype=np.uint8)
    n, N = idx.shape[-3], idx.shape[-1]
    lead = idx.shape[:-3]
    rows = np.zeros(lead + (n, 3, N, row_stride), dtype=np.uint8)
    rows[..., :N] = np.moveaxis(np.asarray(lut, dtype=np.uint8)[idx][..., :3], -1, -3)
    block = np.zeros(lead + (n, agent_stride), dtype=np.uint8)
    block[..., :3 * N * row_stride] = rows.reshape(lead + (n, 3 * N * row_stride))
    return block.reshape(lead + (n * agent_stride,))
