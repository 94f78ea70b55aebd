"""NumPy float32 restatement of per-agent preference sets (extra_args reward_shaping as one dict or a list of one per agent,
``ssd_set_reward_preferences``; DESIGN.md §3 item 20), ``atan2f_ssd`` included.

Every operation below is one float32 NumPy operation, rounded once, in the order of the contract, so the kernel must match it bit
for bit.  A preference set is (alpha, beta, decay, prosocial, svo_angle in radians, svo_weight)."""
import numpy as np

f32 = np.float32
# atan(q) ~ q * P(q^2) on [0, 1]: the coefficients of include/ssd_b200.h (ssd_set_reward_preferences), C0 first, each an exact
# float32 value
ATAN_C = tuple(f32(c) for c in (0.9999961256980896, -0.3331736922264099, 0.19807815551757812, -0.1323334127664566,
                                0.07962366193532944, -0.0336042121052742, 0.006811790633946657))
HALF_PI, PI = f32(np.pi / 2), f32(np.pi)


def atan2f_ssd(y, x):
    """The kernel's fixed float32 atan2 sequence, elementwise.  Signs of zero are not looked at: (±0, x < 0) gives +pi and
    (±0, ±0) gives 0."""
    y, x = np.asarray(y, f32), np.asarray(x, f32)
    ax, ay = np.abs(x), np.abs(y)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    zero = mx == f32(0)
    q = mn / np.where(zero, f32(1), mx)
    s = q * q
    p = np.full_like(q, ATAN_C[-1])
    for c in ATAN_C[-2::-1]:
        p = p * s + c
    t = q * p
    t = np.where(ay > ax, HALF_PI - t, t)
    t = np.where(x < f32(0), PI - t, t)
    t = np.where(y < f32(0), -t, t)
    t = np.where(zero, f32(0), t)
    assert t.dtype == f32
    return t


def host_set(n, alpha, beta, decay, prosocial, svo_angle, svo_weight):
    """(a, b, decay, w, w1, svo, ws) as the host precomputes them in float32 (tests/shaping_ref.py's host_params, plus the
    angle and weight as given)."""
    others = f32(n - 1)
    a = f32(alpha) / others if n > 1 else f32(0)
    b = f32(beta) / others if n > 1 else f32(0)
    return f32(a), f32(b), f32(decay), f32(prosocial), f32(1) - f32(prosocial), f32(svo_angle), f32(svo_weight)


def agent_sets(n_sets, B, n, variant=None, set_of=None):
    """[B, n] set id of every agent: set_of[min(variant[b], n_rows - 1)][i] with a roster (row 0 without ids), else
    min(variant[b], n_sets - 1) (0 without ids)."""
    if set_of is not None:
        set_of = np.asarray(set_of, np.int64).reshape(-1, n)
        row = np.zeros(B, np.int64) if variant is None else np.minimum(np.asarray(variant, np.int64), len(set_of) - 1)
        return set_of[row]
    sid = np.zeros(B, np.int64) if variant is None else np.minimum(np.asarray(variant, np.int64), n_sets - 1)
    return np.repeat(sid[:, None], n, 1)


def pref_step(trace, reward, sets, variant=None, set_of=None, done=None):
    """One step of every env.  trace: float32 [B, n] before the step; reward: int [B, n]; sets: list of preference sets;
    variant: [B] ids or None; set_of: roster [n_rows][n] or None; done: [B] flags of an auto-reset step (their traces restart at
    0) or None.  Returns (shaped, trace after the step), both float32 [B, n]."""
    trace = np.asarray(trace, f32)
    B, n = trace.shape
    table = np.array([host_set(n, *q) for q in sets], dtype=f32)                 # [S, 7]
    a, b, decay, w, w1, svo, ws = (table[agent_sets(len(sets), B, n, variant, set_of), k] for k in range(7))
    r = np.asarray(reward).astype(f32)
    e = trace * decay + r
    c = (np.asarray(reward).astype(np.int64).sum(1).astype(f32) / f32(n))[:, None]
    m = w1 * r + w * c
    D = np.zeros((B, n), f32)
    A = np.zeros((B, n), f32)
    O = np.zeros((B, n), f32)
    lanes = np.arange(n)
    for j in range(n):                                        # ascending j, skipping j == i
        ej = e[:, j:j + 1]
        other = (lanes != j)[None, :]
        D = np.where(other, D + np.maximum(ej - e, f32(0)), D)
        A = np.where(other, A + np.maximum(e - ej, f32(0)), A)
        O = np.where(other, O + ej, O)
    v = np.zeros((B, n), f32)
    if n > 1:
        o = O / f32(n - 1)
        v = np.where(ws != f32(0), ws * np.abs(svo - atan2f_ssd(o, e)), f32(0))
    u = ((m - a * D) - b * A) - v
    if done is not None:
        e = np.where(np.asarray(done, bool)[:, None], f32(0), e)
    assert u.dtype == f32 and e.dtype == f32
    return u, e


class PreferenceRef:
    """The traces of a batch, stepped on the GPU's own rewards, done flags and variant ids."""

    def __init__(self, B, n, sets, variant=None, set_of=None):
        self.sets, self.variant, self.set_of = list(sets), variant, set_of
        self.trace = np.zeros((B, n), f32)
        self.shaped = np.zeros((B, n), f32)

    @classmethod
    def of(cls, env):
        """The restatement of an SSDBatchEnv's preferences: its distinct sets and roster, indexed by its variant ids."""
        var = None if env.variant is None else env.variant.cpu().numpy()
        return cls(env.B, env.n, env.preference_sets, var, env.preference_of)

    def step(self, reward, done=None, envs=slice(None)):
        """A step of envs ``envs`` (a slice); ``done`` only for an auto-reset step."""
        var = None if self.variant is None else np.asarray(self.variant)[envs]
        u, e = pref_step(self.trace[envs], reward[envs], self.sets, var, self.set_of, None if done is None else done[envs])
        self.shaped[envs], self.trace[envs] = u, e

    def reset(self, mask=None):
        if mask is None:
            self.trace[:] = 0
        else:
            self.trace[np.asarray(mask, bool)] = 0
