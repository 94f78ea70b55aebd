"""Plain float64 restatement (NumPy) of the fused observation front end, ``ssd_frontend_forward`` in csrc/frontend_b200.cu:

    u8 agent views (strided planes) -> /256 -> Conv2d(3, 6, 3) + bias -> LeakyReLU -> Flatten (oc, y, x)
                                     -> Linear(6 P^2, 32) -> LeakyReLU                 (P = N - 2, N = 2 view + 1)

``forward64`` is the exact operation, ``forward64_hi_only`` the same with the FC operands rounded to tf32 (what a kernel that
dropped its lo terms would compute), and ``longest_chain`` restates how many tensor-core MMAs the kernel chains on one
accumulator, which is what its error grows with.
"""
import numpy as np

N_OC, N_FEAT = 6, 32


def env_layout(view):
    """The env's own strides (ssd_layout): row stride round4(N), plane stride N * RP, agent stride round16(3 * PS)."""
    N = 2 * view + 1
    RP = (N + 3) // 4 * 4
    PS = N * RP
    return dict(RP=RP, PS=PS, AS=(3 * PS + 15) // 16 * 16)


def gather(buf_u8, rows, AS, PS, RP, view):
    """u8 [rows, 3, N, N] read through the strides, exactly the bytes the kernel addresses."""
    N = 2 * view + 1
    buf = np.ascontiguousarray(np.asarray(buf_u8, dtype=np.uint8).reshape(-1))
    if rows and buf.size < (rows - 1) * AS + 2 * PS + (N - 1) * RP + N:
        raise ValueError("buffer too small for rows x strides")
    return np.lib.stride_tricks.as_strided(buf, (rows, 3, N, N), (AS, PS, RP, 1), writeable=False).copy()


def leaky(v, slope):
    return np.where(v > 0, v, v * slope)


def features64(buf_u8, rows, AS, PS, RP, view, conv_w, conv_b, slope):
    """The FC input: LeakyReLU(conv(obs / 256) + bias) flattened in (oc, y, x) order, float64 [rows, 6 P^2]."""
    P = 2 * view - 1
    x = gather(buf_u8, rows, AS, PS, RP, view).astype(np.float64) / 256
    w = np.asarray(conv_w, dtype=np.float64).reshape(N_OC, 3, 3, 3)
    c = np.broadcast_to(np.asarray(conv_b, dtype=np.float64).reshape(1, N_OC, 1, 1), (rows, N_OC, P, P)).copy()
    for dy in range(3):
        for dx in range(3):
            c += np.einsum("rcyx,oc->royx", x[:, :, dy:dy + P, dx:dx + P], w[:, :, dy, dx])
    return leaky(c, slope).reshape(rows, N_OC * P * P)


def forward64(buf_u8, rows, AS, PS, RP, view, conv_w, conv_b, fc_w, fc_b, slope):
    """Returns (y [rows, 32] float64, M [rows, 32]) with M = |fc_b| + sum_k |W_k| |a_k|, the condition scale of the FC sum."""
    a = features64(buf_u8, rows, AS, PS, RP, view, conv_w, conv_b, slope)
    W = np.asarray(fc_w, dtype=np.float64)
    b = np.asarray(fc_b, dtype=np.float64)
    return leaky(a @ W.T + b, slope), np.abs(a) @ np.abs(W).T + np.abs(b)


def tf32_rna(v):
    """cvt.rna.tf32.f32 (and the host's host_tf32): to float32, then nearest with 10 mantissa bits, ties away from zero."""
    bits = np.asarray(v, dtype=np.float32).view(np.uint32)
    return ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def forward64_hi_only(buf_u8, rows, AS, PS, RP, view, conv_w, conv_b, fc_w, fc_b, slope):
    """forward64 with both FC operands rounded to tf32 (the hi*hi product alone), summed in float64."""
    a = tf32_rna(features64(buf_u8, rows, AS, PS, RP, view, conv_w, conv_b, slope)).astype(np.float64)
    W = tf32_rna(np.asarray(fc_w, dtype=np.float32)).astype(np.float64)
    return leaky(a @ W.T + np.asarray(fc_b, dtype=np.float64), slope)


def longest_chain(view):
    """Most MMAs the kernel chains on one hi*hi TMEM accumulator in a segment that covers a whole tile: a tile is P * XB chunks
    of 2 stages (kStagesPerChunk), a stage is 6 K=8 steps shared by 2 issuers, and each issuer rotates its steps over
    rotation() = min(7, ceil(steps / 24)) accumulators."""
    P = 2 * view - 1
    chunks = P * ((P + 15) // 16)
    steps = chunks * 2 * 6 // 2
    n_rot = min(7, (steps + 23) // 24)
    return -(-steps // n_rot)


def tolerance(view):
    """Bound on |got - y64| / (1 + |y64|): 1e-6 for chains up to the 50 MMAs of V=15, growing linearly with the chain beyond."""
    return 1e-6 * max(1.0, longest_chain(view) / 50)


def rel_err(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return float((np.abs(got - want) / (1 + np.abs(want))).max()) if got.size else 0.0
