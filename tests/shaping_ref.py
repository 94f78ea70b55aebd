"""NumPy float32 restatement of the shaped reward (extra_args reward_shaping, ``ssd_set_reward_shaping``; DESIGN.md §3 item 17).

Every operation below is one float32 NumPy operation, rounded once, in the order of the contract, so the kernel must match it bit
for bit.  ``shape64`` evaluates the same formulas in float64 (no intermediate rounding) for the CPU check of the restatement."""
import numpy as np

f32 = np.float32
DEFAULT_DECAY = float(f32(0.99 * 0.975))


def host_params(n, alpha, beta, decay, prosocial):
    """(a, b, decay, w, w1) as the host precomputes them in float32: a = alpha/(n-1), b = beta/(n-1) (0 for n = 1), w1 = 1 - w."""
    others = f32(n - 1)
    a = f32(alpha) / others if n > 1 else f32(0)
    b = f32(beta) / others if n > 1 else f32(0)
    return f32(a), f32(b), f32(decay), f32(prosocial), f32(1) - f32(prosocial)


def env_params(params, n, B, variant=None):
    """Per-env float32 [B] arrays a, b, decay, w, w1: params[0] for every env, or params[min(variant[b], len(params) - 1)]."""
    table = np.array([host_params(n, *q) for q in params], dtype=f32)              # [P, 5]
    pid = np.zeros(B, np.int64) if variant is None else np.minimum(np.asarray(variant, np.int64), len(params) - 1)
    return [table[pid, k] for k in range(5)]


def shape_step(trace, reward, params, variant=None, done=None):
    """One step of every env.  trace: float32 [B, n] before the step; reward: int [B, n]; params: list of (alpha, beta, decay,
    prosocial); variant: [B] ids or None; done: [B] flags of an auto-reset step (their traces restart at 0) or None.
    Returns (shaped, trace after the step), both float32 [B, n]."""
    trace = np.asarray(trace, f32)
    B, n = trace.shape
    a, b, decay, w, w1 = (x[:, None] for x in env_params(params, n, B, variant))
    r = np.asarray(reward).astype(f32)
    e = trace * decay + r
    c = (np.asarray(reward).astype(np.int64).sum(1).astype(f32) / f32(n))[:, None]
    m = w1 * r + w * c
    D = np.zeros((B, n), f32)
    A = np.zeros((B, n), f32)
    lanes = np.arange(n)
    for j in range(n):                                        # ascending j, skipping j == i
        ej = e[:, j:j + 1]
        other = (lanes != j)[None, :]
        D = np.where(other, D + np.maximum(ej - e, f32(0)), D)
        A = np.where(other, A + np.maximum(e - ej, f32(0)), A)
    u = (m - a * D) - b * A
    if done is not None:
        e = np.where(np.asarray(done, bool)[:, None], f32(0), e)
    assert u.dtype == f32 and e.dtype == f32
    return u, e


def shape64(trace, reward, params, variant=None):
    """The same step in float64 from the float32 parameters and trace: (shaped, trace after), float64 [B, n]."""
    trace = np.asarray(trace, np.float64)
    B, n = trace.shape
    pid = np.zeros(B, np.int64) if variant is None else np.minimum(np.asarray(variant, np.int64), len(params) - 1)
    q = np.array([[float(f32(x)) for x in p] for p in params])[pid]
    alpha, beta, decay, w = (q[:, k:k + 1] for k in range(4))
    r = np.asarray(reward, np.float64)
    e = trace * decay + r
    c = r.sum(1, keepdims=True) / n
    gap = e[:, None, :] - e[:, :, None]                       # [b, i, j] = e_j - e_i
    D = np.maximum(gap, 0).sum(2)
    A = np.maximum(-gap, 0).sum(2)
    k = 1.0 / (n - 1) if n > 1 else 0.0
    return (1 - w) * r + w * c - alpha * k * D - beta * k * A, e


class ShapingRef:
    """The traces of a batch, stepped on the GPU's own rewards, done flags and variant ids."""

    def __init__(self, B, n, params, variant=None):
        self.params, self.variant = list(params), variant
        self.trace = np.zeros((B, n), f32)
        self.shaped = np.zeros((B, n), f32)

    def step(self, reward, done=None, envs=slice(None)):
        """A step of envs ``envs`` (a slice); ``done`` only for an auto-reset step."""
        var = None if self.variant is None else np.asarray(self.variant)[envs]
        u, e = shape_step(self.trace[envs], reward[envs], self.params, var, None if done is None else done[envs])
        self.shaped[envs], self.trace[envs] = u, e

    def reset(self, mask=None):
        if mask is None:
            self.trace[:] = 0
        else:
            self.trace[np.asarray(mask, bool)] = 0
